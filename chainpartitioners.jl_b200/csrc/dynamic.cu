// dynamic.cu -- kernel family "dp_layer": DynamicBottleneckSplitter / DynamicTotalSplitter
// (DynamicSplitter.jl:15-50; also the Reference*Splitter ground truth, ReferenceSplitter.jl:1-13).
//
//   cst[j', 1] = c(1, j', 1)
//   cst[j', k] = min_j g(cst[j, k-1], c(j, j', k)),   g = max (bottleneck) or + (total),
//   ties -> the LARGEST j (the reference updates on `<=`, DynamicSplitter.jl:40).
//
// One launch per layer k, one thread (bottleneck) or one warp/CTA (total) per j'.  For monotone
// costs (beta >= 0, asserted by the reference's bound_stripe) the bottleneck recurrence needs no
// scan over j: f_{k-1}(j) is non-decreasing and c(j, j') non-increasing in j, so the minimum sits at
// their crossing, found by binary search; the reference's rightmost tie is recovered by a second
// binary search on the previous row (SURVEY.md section 7 "hard parts", re-verified in tests).
#include <algorithm>
#include "engine.cuh"

namespace cpb {

template <class T>
__global__ void __launch_bounds__(256) k_dp_first(const __grid_constant__ DevOracle o, T* __restrict__ cst, u32* __restrict__ ptr) {
  const u32 n1 = o.n + 1;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < n1; t += stride) {
    const u32 jp = (u32)t + 1;
    cst[jp] = dev_cost<T>(o, 1, jp);
    ptr[jp] = 1;
  }
}

// bottleneck layer: a(j) = prev[j] (non-decreasing), b(j) = c(j, j') (non-increasing)
template <class T>
__global__ void __launch_bounds__(256) k_dp_bottleneck(const __grid_constant__ DevOracle o, const T* __restrict__ prev, T* __restrict__ cur,
                                                       u32* __restrict__ ptr, u32 jp_first, u32 k) {
  const u32 n1 = o.n + 1;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x + jp_first; t <= n1; t += stride) {
    const u32 jp = (u32)t;
    // j* = min{ j in [1, jp] : a(j) >= b(j) }, jp + 1 if none
    u32 lo = 1, hi = jp + 1;
    while (lo < hi) {
      const u32 mid = lo + ((hi - lo) >> 1);
      if (prev[mid] >= dev_cost<T>(o, mid, jp, k)) hi = mid; else lo = mid + 1;
    }
    const u32 js = lo;
    T v;
    u32 arg;
    if (js > jp) {  // a < b everywhere: h = b is minimised at the right end
      arg = jp;
      v = dev_cost<T>(o, jp, jp, k);
    } else {
      const T va = prev[js];
      bool right = true;
      T vb = va;
      if (js > 1) {
        vb = dev_cost<T>(o, js - 1, jp, k);
        right = va <= vb;
      }
      if (right) {
        v = va;
        // largest j in [js, jp] with a(j) <= v
        u32 l2 = js, h2 = jp;
        while (l2 < h2) {
          const u32 mid = l2 + ((h2 - l2 + 1) >> 1);
          if (prev[mid] <= v) l2 = mid; else h2 = mid - 1;
        }
        arg = l2;
      } else {
        v = vb;
        arg = js - 1;
      }
    }
    cur[jp] = v;
    ptr[jp] = arg;
  }
}

// Tie rules of the total-cost layers.  TIE_RIGHT: DynamicTotalSplitter -- the largest j in [1, j'] among the minimisers
// (`<=` while scanning upwards, DynamicSplitter.jl:40).  TIE_CONVEX: ConvexTotalSplitter (ConvexTotalChunker.jl:26-55) --
// the row starts from the empty last part (ptr = j', :47-50) and chunk_convex! then overrides it on `<=` with its
// candidate, which for costs obeying the quadrangle inequality (:121) is the SMALLEST minimiser in [1, j' - 1]
// (SURVEY.md App. B, re-verified against the stack algorithm in tests/test_oracle_solvers.py).
enum { TIE_RIGHT = 0, TIE_CONVEX = 1 };
template <int TIE, class T> __device__ __forceinline__ bool tie_better(T ob, u32 oa, T best, u32 arg) {
  if (oa == 0) return false;
  if (arg == 0 || ob < best) return true;
  return ob == best && (TIE == TIE_RIGHT ? oa > arg : oa < arg);
}

// total layer, one warp per j': scan of all j in [1, j'] with a rightmost-argmin reduction.
// (O(n^2) oracle queries per layer; the monotone divide & conquer version replaces it for large n.)
// MAXOP: the bottleneck recurrence (g = max) for costs the crossing search of k_dp_bottleneck cannot take (decreasing
// secondary costs): the same exhaustive scan, O(n^2) queries per layer.
template <int TIE, class T, bool MAXOP = false>
__global__ void __launch_bounds__(256) k_dp_total(const __grid_constant__ DevOracle o, const T* __restrict__ prev, T* __restrict__ cur,
                                                  u32* __restrict__ ptr, u32 jp_first, u32 k) {
  const u32 n1 = o.n + 1;
  const int lane = threadIdx.x & 31;
  const size_t warps = ((size_t)gridDim.x * blockDim.x) >> 5;
  for (size_t t = (((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) + jp_first; t <= n1; t += warps) {
    const u32 jp = (u32)t;
    T best = 0;
    u32 arg = 0;
    const u32 j_last = TIE == TIE_RIGHT ? jp : jp - 1;
    for (u32 j = 1 + lane; j <= j_last; j += 32) {
      const T cj = dev_cost<T>(o, j, jp, k);
      const T c = MAXOP ? max(prev[j], cj) : prev[j] + cj;
      // ascending j within a lane: `<=` keeps the largest minimiser, `<` the smallest
      if (arg == 0 || (TIE == TIE_RIGHT ? c <= best : c < best)) { best = c; arg = j; }
    }
    for (int off = 16; off > 0; off >>= 1) {
      const T ob = __shfl_down_sync(0xffffffffu, best, off);
      const u32 oa = __shfl_down_sync(0xffffffffu, arg, off);
      if (tie_better<TIE>(ob, oa, best, arg)) { best = ob; arg = oa; }
    }
    if (lane == 0) {
      if (TIE == TIE_CONVEX) {  // the empty last part stays only if it is strictly cheaper
        const T init = prev[jp] + dev_cost<T>(o, jp, jp, k);
        if (arg == 0 || init < best) { best = init; arg = jp; }
      }
      cur[jp] = best;
      ptr[jp] = arg;
    }
  }
}

// total layer by monotone divide & conquer.  For Monge ("convex", ConvexTotalChunker.jl:121) costs the
// rightmost argmin opt(j') is non-decreasing in j' (SURVEY.md App. B / E8), so the candidates of the
// midpoint of a segment are bounded by the argmins of its already solved neighbours.  One launch per
// level of the implicit balanced tree over t = j' - 1 in [0, n]; one CTA per node scans its candidate
// range with a rightmost-argmin reduction.  Total work per layer O(n log n) oracle queries.
template <int TIE, class T>
__global__ void __launch_bounds__(256) k_dp_total_dc(const __grid_constant__ DevOracle o, const T* __restrict__ prev, T* __restrict__ cur,
                                                     u32* __restrict__ ptr, u32 step, u32 first_t, u32 t_stride, u32 k) {
  __shared__ T s_best[8];
  __shared__ u32 s_arg[8];
  const u32 n = o.n;
  const u64 t64 = (u64)first_t + (u64)blockIdx.x * t_stride;
  if (t64 > n) return;
  const u32 t = (u32)t64;
  const u32 jp = t + 1;
  u32 lo = 1, hi = jp;
  if (step > 0) {  // neighbours t - step and min(t + step, n) are solved
    lo = ptr[t - step + 1];
    hi = min(hi, ptr[min(t + step, n) + 1]);
  }
  T best = 0;
  u32 arg = 0;
  const u32 j_last = TIE == TIE_RIGHT ? hi : min(hi, jp - 1);
  for (u32 j = lo + threadIdx.x; j <= j_last; j += blockDim.x) {
    const T c = prev[j] + dev_cost<T>(o, j, jp, k);
    if (arg == 0 || (TIE == TIE_RIGHT ? c <= best : c < best)) { best = c; arg = j; }
  }
  for (int off = 16; off > 0; off >>= 1) {
    const T ob = __shfl_down_sync(0xffffffffu, best, off);
    const u32 oa = __shfl_down_sync(0xffffffffu, arg, off);
    if (tie_better<TIE>(ob, oa, best, arg)) { best = ob; arg = oa; }
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) { s_best[w] = best; s_arg[w] = arg; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 1; k < 8; ++k) {
      const T ob = s_best[k];
      const u32 oa = s_arg[k];
      if (tie_better<TIE>(ob, oa, best, arg)) { best = ob; arg = oa; }
    }
    if (TIE == TIE_CONVEX && hi == jp) {  // the empty last part (candidate j') stays only if it is strictly cheaper
      const T init = prev[jp] + dev_cost<T>(o, jp, jp, k);
      if (arg == 0 || init < best) { best = init; arg = jp; }
    }
    cur[jp] = best;
    ptr[jp] = arg;
  }
}

// weight-constrained layer (DynamicSplitter.jl:206-247) for weights w(j, j') = a + b_v (j' - j) + b_p (pos[j'] - pos[j])
// with b_v, b_p >= 0: the feasible predecessors of j' are the window [max(lo_prev, j0(j')), min(j', hi_prev)], j0(j') the
// smallest j with w(j, j') <= w_max (the reference advances j0 monotonically, :231-233; here a binary search, or
// j' - W when there is no pin term); rightmost argmin (`<=`).  A count weight (weights.cu) hands j0(j') over as the window
// array first_fit (nullptr: the affine weight).
struct DevWeight {
  i64 a, bv, bp, w_max;
  const u32* first_fit;
};
__device__ __forceinline__ bool weight_ok(const DevOracle& o, const DevWeight& w, u32 j, u32 jp) {
  return w.a + (i64)(jp - j) * w.bv + ((i64)__ldg(o.pos + (jp - 1)) - (i64)__ldg(o.pos + (j - 1))) * w.bp <= w.w_max;
}
template <class T>
__global__ void __launch_bounds__(256) k_dp_constrained(const __grid_constant__ DevOracle o, const T* __restrict__ prev, T* __restrict__ cur,
                                                        u32* __restrict__ ptr, int total, u32 lo_k, u32 hi_k, u32 lo_p, u32 hi_p, u32 W, int first,
                                                        DevWeight wt, u32 k) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x + lo_k; t <= hi_k; t += stride) {
    const u32 jp = (u32)t;
    if (first) {  // k = 1: cst[j', 1] = f(1, j', 1)
      cur[jp] = dev_cost<T>(o, 1, jp);
      ptr[jp] = 1;
      continue;
    }
    u32 j0 = max(lo_p, jp > W ? jp - W : 1u);
    const u32 j1 = min(jp, hi_p);
    if (wt.first_fit) {
      j0 = max(j0, __ldg(wt.first_fit + jp));
    } else if (wt.bp != 0) {  // smallest j in [j0, jp] with w(j, j') <= w_max (w shrinks as j grows)
      u32 a = j0, b = jp;
      while (a < b) {
        const u32 mid = a + ((b - a) >> 1);
        if (weight_ok(o, wt, mid, jp)) b = mid; else a = mid + 1;
      }
      j0 = a;
    }
    T best = 0;
    u32 arg = 0;
    for (u32 j = j0; j <= j1; ++j) {
      const T c = dev_cost<T>(o, j, jp, k);
      const T v = total ? prev[j] + c : max(prev[j], c);
      if (arg == 0 || v <= best) { best = v; arg = j; }
    }
    cur[jp] = best;
    ptr[jp] = arg;
  }
}

// the same layer with one warp per j' for wide windows (a thread-per-j' scan of thousands of split points is one dependent
// chain of oracle queries per thread and leaves most of the machine idle): lanes share the window, butterfly reduction to the
// smallest value and, among ties, the largest column (the `<=` rule)
template <class T>
__global__ void __launch_bounds__(256) k_dp_constrained_warp(const __grid_constant__ DevOracle o, const T* __restrict__ prev, T* __restrict__ cur,
                                                             u32* __restrict__ ptr, int total, u32 lo_k, u32 hi_k, u32 lo_p, u32 hi_p, u32 W, DevWeight wt, u32 k) {
  const int lane = threadIdx.x & 31;
  const size_t warps = ((size_t)gridDim.x * blockDim.x) >> 5;
  for (size_t t = (((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) + lo_k; t <= hi_k; t += warps) {
    const u32 jp = (u32)t;
    u32 j0 = max(lo_p, jp > W ? jp - W : 1u);
    const u32 j1 = min(jp, hi_p);
    if (wt.first_fit) {
      j0 = max(j0, __ldg(wt.first_fit + jp));
    } else if (wt.bp != 0) {
      u32 a = j0, b = jp;
      while (a < b) {
        const u32 mid = a + ((b - a) >> 1);
        if (weight_ok(o, wt, mid, jp)) b = mid; else a = mid + 1;
      }
      j0 = a;
    }
    T best = 0;
    u32 arg = 0;
    for (u64 j64 = (u64)j0 + lane; j64 <= j1; j64 += 32) {
      const u32 j = (u32)j64;
      const T c = dev_cost<T>(o, j, jp, k);
      const T v = total ? prev[j] + c : max(prev[j], c);
      if (arg == 0 || v <= best) { best = v; arg = j; }
    }
    for (int d = 16; d > 0; d >>= 1) {
      const T ov = __shfl_xor_sync(0xffffffffu, best, d);
      const u32 oa = __shfl_xor_sync(0xffffffffu, arg, d);
      if (oa != 0 && (arg == 0 || ov < best || (ov == best && oa > arg))) { best = ov; arg = oa; }
    }
    if (lane == 0) {
      cur[jp] = best;
      ptr[jp] = arg;
    }
  }
}

__global__ void k_dp_unravel(const u32* __restrict__ ptr, u32 n2, int K, u32 n1, i64* __restrict__ spl) {
  // DynamicSplitter.jl:89-99
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    spl[K] = n1;
    for (int k = K; k >= 1; --k) spl[k - 1] = ptr[(size_t)(k - 1) * n2 + (u32)spl[k]];
  }
}

template <class T, int TIE> static void dynamic_T(Oracle& f, bool total, i64 K, int64_t* h_spl_out) {
  const Matrix& A = *f.A;
  const u32 n1 = (u32)A.n + 1, n2 = n1 + 1;
  CPB_REQUIRE((double)K * n2 * 4.0 < 64e9, "DP pointer table would not fit");
  ProfScope prof("dp_layer");
  // Monge cost models with non-negative betas: monotone rightmost argmin (see k_dp_total_dc)
  bool monge = f.mdl.kind == CPB_MODEL_WORK || f.mdl.kind == CPB_MODEL_CONNECTIVITY || f.mdl.kind == CPB_MODEL_MONOSYM;
  for (int t = 1; t <= 3; ++t) monge = monge && f.mdl.coef[t] >= 0;
  DBuf<T> rowa(n2), rowb(n2);
  DBuf<u32> ptr((size_t)K * n2);
  DBuf<i64> spl(K + 1);
  const unsigned grid = (unsigned)std::min<size_t>(((size_t)n1 + 255) / 256, (size_t)ctx().sm_count * 8);
  CPB_LAUNCH(k_dp_first<T>, grid, 256, 0, f.dev, rowa.get(), ptr.get());
  T* prev = rowa.get();
  T* cur = rowb.get();
  for (i64 k = 2; k <= K; ++k) {
    const u32 jp_first = (k == K) ? n1 : 1;  // DynamicSplitter.jl:34
    u32* p = ptr.get() + (size_t)(k - 1) * n2;
    if (!total && (f.mdl.kind == CPB_MODEL_SECCONN || f.mdl.kind == CPB_MODEL_SECEDGE)) {  // decreasing costs: exhaustive scan with g = max
      const size_t rows = (size_t)n1 - jp_first + 1;
      const unsigned g = (unsigned)std::min<size_t>((rows * 32 + 255) / 256, (size_t)ctx().sm_count * 8);
      CPB_LAUNCH((k_dp_total<TIE_RIGHT, T, true>), g, 256, 0, f.dev, prev, cur, p, jp_first, (u32)k);
    } else if (!total) {
      const unsigned g = (k == K) ? 1 : grid;
      CPB_LAUNCH(k_dp_bottleneck<T>, g, 256, 0, f.dev, prev, cur, p, jp_first, (u32)k);
    } else if (monge && A.n > 64) {
      const u32 n = (u32)A.n;
      // j' = n + 1 (t = n): full scan; the only point the last layer needs (DynamicSplitter.jl:34)
      CPB_LAUNCH((k_dp_total_dc<TIE, T>), 1, 256, 0, f.dev, prev, cur, p, 0u, n, 1u, (u32)k);
      if (k < K) {
        CPB_LAUNCH((k_dp_total_dc<TIE, T>), 1, 256, 0, f.dev, prev, cur, p, 0u, 0u, 1u, (u32)k);  // j' = 1 (t = 0)
        u32 D = 1;
        while (((u64)1 << D) <= n) ++D;  // 2^D > n
        for (u32 step = (u32)1 << (D - 1); step >= 1; step >>= 1) {
          // nodes t = step * (2 i + 1) <= n, t != n (already solved)
          const u64 nodes = ((u64)n / step + 1) / 2;
          if (nodes > 0) CPB_LAUNCH((k_dp_total_dc<TIE, T>), (unsigned)nodes, 256, 0, f.dev, prev, cur, p, step, step, 2 * step, (u32)k);
        }
      }
    } else {
      const size_t rows = (size_t)n1 - jp_first + 1;
      const unsigned g = (unsigned)std::min<size_t>((rows * 32 + 255) / 256, (size_t)ctx().sm_count * 8);
      CPB_LAUNCH((k_dp_total<TIE, T>), g, 256, 0, f.dev, prev, cur, p, jp_first, (u32)k);
    }
    std::swap(prev, cur);
  }
  CPB_LAUNCH(k_dp_unravel, 1, 32, 0, ptr.get(), n2, (int)K, n1, spl.get());
  CPB_CUDA(cudaMemcpyAsync(h_spl_out, spl.get(), (K + 1) * sizeof(i64), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
}

template <class T> static void dynamic_constrained_T(Oracle& f, bool total, const Windows& win, i64 K, int64_t* h_spl_out) {
  const Matrix& A = *f.A;
  const i64 n = A.n;
  std::vector<i64> lo, hi;
  if (!column_constraints(win, n, K, lo, hi)) {  // :217-222 infeasible -> degenerate partition
    degenerate_partition(n, K, h_spl_out);
    return;
  }
  const i64 W = win.W;
  const DevWeight dw{win.a, win.bv, win.bp, win.w_max, win.first_fit.get()};
  const u32 n1 = (u32)n + 1, n2 = n1 + 1;
  ProfScope prof("dp_layer");
  DBuf<T> rowa(n2), rowb(n2);
  DBuf<u32> ptr((size_t)K * n2);
  DBuf<i64> spl(K + 1);
  ptr.zero();
  T* prev = rowa.get();
  T* cur = rowb.get();
  for (i64 k = 1; k <= K; ++k) {
    const size_t cnt = (size_t)(hi[k] - lo[k] + 1);
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>((cnt + 255) / 256, (size_t)ctx().sm_count * 8));
    const bool wide = k > 1 && std::min<i64>(W, hi[k - 1] - lo[k - 1] + 1) > 64 && std::getenv("CPB_DP_THREAD_WINDOWS") == nullptr;
    if (wide) {
      const unsigned wgrid = (unsigned)std::max<size_t>(1, std::min<size_t>((cnt * 32 + 255) / 256, (size_t)ctx().sm_count * 16));
      CPB_LAUNCH(k_dp_constrained_warp<T>, wgrid, 256, 0, f.dev, prev, cur, ptr.get() + (size_t)(k - 1) * n2, total ? 1 : 0, (u32)lo[k], (u32)hi[k],
                 (u32)lo[k - 1], (u32)hi[k - 1], (u32)std::min<i64>(std::max<i64>(W, 0), n + 1), dw, (u32)k);
    } else {
      CPB_LAUNCH(k_dp_constrained<T>, grid, 256, 0, f.dev, prev, cur, ptr.get() + (size_t)(k - 1) * n2, total ? 1 : 0, (u32)lo[k], (u32)hi[k],
                 (u32)(k > 1 ? lo[k - 1] : 1), (u32)(k > 1 ? hi[k - 1] : 1), (u32)std::min<i64>(std::max<i64>(W, 0), n + 1), k == 1 ? 1 : 0,
                 dw, (u32)k);
    }
    std::swap(prev, cur);
  }
  CPB_LAUNCH(k_dp_unravel, 1, 32, 0, ptr.get(), n2, (int)K, n1, spl.get());
  CPB_CUDA(cudaMemcpyAsync(h_spl_out, spl.get(), (K + 1) * sizeof(i64), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
}

// ---- ConvexTotalSplitter{<:ConstrainedCost} (ConvexTotalChunker.jl:167-265) ---------------------------------------------
// Per layer the reference runs chunk_convex_constrained! on window-constrained columns of Extended costs: the columns
// after J0 = j'_lo[k-1] fall into blocks (b_t, b_t+1], b_t+1 = the last column that still fits into one part with b_t; a
// block first receives, from the "staircase" pass, the best split point among the previous block (the reversed indices of
// :252-258 make it the RIGHTMOST minimiser, and the value replaces the layer's initial empty-part candidate), then the
// in-block pass offers the LEFTMOST minimiser of [b_t, j'-1] and wins ties (`<=`, :66,74).  Block 0 only has the in-block
// pass against the empty-part initialisation.  The values are the constrained optimum; this rule reproduces the pointers:
// 2500/2500 random cases (vertex- and pin-weighted windows, Int64 and Float64 costs) against the restated algorithm
// (tools/convex_k_rule.py), and tests/test_gpu_parity.py::test_constrained_convex_total_splitter.
// Every split point of the window is evaluated (O(n W) queries).  A per-block divide & conquer over "monotone" minimisers was
// tried (3-7 ms instead of 80-118 ms at n = 2^14, W = 1.5 n / K) and is WRONG: these costs obey the INVERSE quadrangle
// inequality -- the reason the reference uses a stack -- and inside a constrained block the minimisers are not monotone
// (3 of ~230 random cases differed, one with a worse total).  Dropped; see profiles/r01_next.md.
template <class T> struct DpInf;
template <> struct DpInf<i64> { static __device__ __forceinline__ i64 get() { return (i64)1 << 61; } };
template <> struct DpInf<double> { static __device__ __forceinline__ double get() { return 1e300; } };

template <class T>
__global__ void __launch_bounds__(256) k_dp_convex_constrained(const __grid_constant__ DevOracle o, const T* __restrict__ prev, T* __restrict__ cur,
                                                               u32* __restrict__ ptr, u32 lo_k, u32 hi_k, u32 lo_p, u32 hi_p, DevWeight wt, u32 k,
                                                               const u32* __restrict__ blk, u32 nblk) {
  // one warp per j': the lanes share the window (wide windows -- w_max = 1.5 n / K in the reference's table -- would leave a
  // thread-per-j' layer with a few thousand dependent query chains per thread and most of the machine idle)
  const T INF = DpInf<T>::get();
  const int lane = threadIdx.x & 31;
  const size_t warps = ((size_t)gridDim.x * blockDim.x) >> 5;
  for (size_t idx = (((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) + lo_k; idx <= hi_k; idx += warps) {
    const u32 jp = (u32)idx;
    // the layer's initialisation: the empty part k (ptr = j')
    T best = (jp >= lo_p && jp <= hi_p && prev[jp] < INF) ? prev[jp] + dev_cost<T>(o, jp, jp, k) : INF;
    u32 arg = jp;
    if (jp > blk[0]) {
      u32 a = 0, b = nblk;  // largest t with blk[t] < jp   (blk[0] < jp <= blk[nblk])
      while (b - a > 1) {
        const u32 mid = a + ((b - a) >> 1);
        if (__ldg(blk + mid) < jp) a = mid; else b = mid;
      }
      const u32 j0 = __ldg(blk + a);
      if (a > 0) {  // staircase pass: rightmost minimiser among the previous block's columns that still fit; replaces the initialisation
        u32 lo_j = __ldg(blk + a - 1) + 1;
        const u32 hi_j = min(j0, hi_p);
        if (wt.first_fit) {  // the same smallest fitting j, read from the window array
          lo_j = max(max(lo_j, __ldg(wt.first_fit + jp)), lo_p);
        } else {
          u32 x = lo_j, y = j0;  // smallest j in [lo_j, j0] with w(j, j') <= w_max (j0 itself fits: j' lies in its block)
          while (x < y) {
            const u32 mid = x + ((y - x) >> 1);
            if (weight_ok(o, wt, mid, jp)) y = mid; else x = mid + 1;
          }
          lo_j = max(x, lo_p);
        }
        T vb = INF;
        u32 ab = 0;
        for (u64 j64 = (u64)lo_j + lane; j64 <= hi_j; j64 += 32) {
          const u32 j = (u32)j64;
          const T pv = prev[j];
          if (pv >= INF) continue;
          const T v = pv + dev_cost<T>(o, j, jp, k);
          if (ab == 0 || v <= vb) { vb = v; ab = j; }
        }
        for (int d = 16; d > 0; d >>= 1) {  // smallest value, then the largest column
          const T ov = __shfl_xor_sync(0xffffffffu, vb, d);
          const u32 oa = __shfl_xor_sync(0xffffffffu, ab, d);
          if (oa != 0 && (ab == 0 || ov < vb || (ov == vb && oa > ab))) { vb = ov; ab = oa; }
        }
        best = ab ? vb : INF;
        arg = ab ? ab : j0;
      }
      // in-block pass: leftmost minimiser of [j0, j'-1]; wins ties against what the column holds
      T vin = INF;
      u32 jin = 0;
      for (u64 j64 = (u64)max(j0, lo_p) + lane; j64 <= min(jp - 1, hi_p); j64 += 32) {
        const u32 j = (u32)j64;
        const T pv = prev[j];
        if (pv >= INF) continue;
        const T v = pv + dev_cost<T>(o, j, jp, k);
        if (jin == 0 || v < vin) { vin = v; jin = j; }
      }
      for (int d = 16; d > 0; d >>= 1) {  // smallest value, then the smallest column
        const T ov = __shfl_xor_sync(0xffffffffu, vin, d);
        const u32 oa = __shfl_xor_sync(0xffffffffu, jin, d);
        if (oa != 0 && (jin == 0 || ov < vin || (ov == vin && oa < jin))) { vin = ov; jin = oa; }
      }
      if (jin != 0 && (best >= INF || vin <= best)) { best = vin; arg = jin; }
    }
    if (lane == 0) {
      cur[jp] = best;
      ptr[jp] = arg;
    }
  }
}

template <class T> static void convex_constrained_T(Oracle& f, const Windows& win, i64 K, int64_t* h_spl_out) {
  const Matrix& A = *f.A;
  const i64 n = A.n;
  std::vector<i64> lo, hi;
  if (!column_constraints(win, n, K, lo, hi)) {  // ConvexTotalChunker.jl:184-189 infeasible -> degenerate partition
    degenerate_partition(n, K, h_spl_out);
    return;
  }
  const DevWeight dw{win.a, win.bv, win.bp, win.w_max, win.first_fit.get()};
  const u32 n1 = (u32)n + 1, n2 = n1 + 1;
  ProfScope prof("dp_layer");
  DBuf<T> rowa(n2), rowb(n2);
  DBuf<u32> ptr((size_t)K * n2), dblk(n2);
  DBuf<i64> spl(K + 1);
  ptr.zero();
  T* prev = rowa.get();
  T* cur = rowb.get();
  std::vector<u32> blk;
  for (i64 k = 1; k <= K; ++k) {
    const size_t cnt = (size_t)(hi[k] - lo[k] + 1);
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>((cnt + 255) / 256, (size_t)ctx().sm_count * 8));
    if (k == 1) {
      CPB_LAUNCH(k_dp_constrained<T>, grid, 256, 0, f.dev, prev, cur, ptr.get(), 1, (u32)lo[1], (u32)hi[1], 1u, 1u, 0u, 1, dw, 1u);
    } else {
      // the block chain of this layer: b_0 = j'_lo[k-1], b_1 = the reach of b_0 (at least b_0 + 1, :213-216), b_t+1 = the reach of b_t
      const i64 J0 = lo[k - 1], JP1 = hi[k];
      blk.clear();
      blk.push_back((u32)J0);
      for (i64 b = J0; b < JP1;) {
        const i64 nx = std::max(win.reach(b, JP1), b + 1);
        blk.push_back((u32)nx);
        b = nx;
      }
      CPB_CUDA(cudaMemcpyAsync(dblk.get(), blk.data(), blk.size() * sizeof(u32), cudaMemcpyHostToDevice, ctx().stream));
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));  // blk is reused by the next layer
      const unsigned wgrid = (unsigned)std::max<size_t>(1, std::min<size_t>((cnt * 32 + 255) / 256, (size_t)ctx().sm_count * 16));
      CPB_LAUNCH(k_dp_convex_constrained<T>, wgrid, 256, 0, f.dev, prev, cur, ptr.get() + (size_t)(k - 1) * n2, (u32)lo[k], (u32)hi[k], (u32)lo[k - 1],
                 (u32)hi[k - 1], dw, (u32)k, dblk.get(), (u32)(blk.size() - 1));
    }
    std::swap(prev, cur);
  }
  CPB_LAUNCH(k_dp_unravel, 1, 32, 0, ptr.get(), n2, (int)K, n1, spl.get());
  CPB_CUDA(cudaMemcpyAsync(h_spl_out, spl.get(), (K + 1) * sizeof(i64), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
}

void solve_dynamic(Oracle& f, bool total, const cpb_constraint* con, i64 K, int64_t* h_spl_out) {
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  if (con && con->enabled) {
    if (f.dev.kind == CPB_MODEL_BLOCK || f.dev.kind == CPB_MODEL_COLBLOCK)
      throw Error(CPB_ERR_UNSUPPORTED, "dynamic splitters need an affine random-access oracle");
    const Windows win = windows_affine(*f.A, con);
    oracle_ensure_ranks(f);
    if (f.dev.is_float) dynamic_constrained_T<double>(f, total, win, K, h_spl_out); else dynamic_constrained_T<i64>(f, total, win, K, h_spl_out);
    return;
  }
  if (f.dev.kind == CPB_MODEL_BLOCK || f.dev.kind == CPB_MODEL_COLBLOCK)
    throw Error(CPB_ERR_UNSUPPORTED, "dynamic splitters need an affine random-access oracle");
  if (!total && f.mdl.kind != CPB_MODEL_SECCONN && f.mdl.kind != CPB_MODEL_SECEDGE) {
    // the crossing search needs monotone costs: the same beta >= 0 the reference asserts in bound_stripe
    for (int t = 1; t <= 4; ++t)
      if (f.mdl.coef[t] < 0 && !(f.mdl.kind == CPB_MODEL_MONOSYM && t == 4))
        throw Error(CPB_ERR_UNSUPPORTED, "bottleneck DP on the device needs non-negative beta coefficients");
    if (f.mdl.kind == CPB_MODEL_SYMCONN || f.mdl.kind == CPB_MODEL_HYPEREDGE || f.mdl.kind == CPB_MODEL_SYMEDGECUT)
      throw Error(CPB_ERR_UNSUPPORTED, "bottleneck DP on the device needs a monotone cost model");
  }
  oracle_ensure_ranks(f);
  if (f.dev.is_float) dynamic_T<double, TIE_RIGHT>(f, total, K, h_spl_out); else dynamic_T<i64, TIE_RIGHT>(f, total, K, h_spl_out);
}

// partition_stripe(A, K, DynamicBottleneck/TotalSplitter(ConstrainedCost(f, w, w_max))) with a count weight w: the same layers,
// the windows from w's window array
void solve_dynamic_weighted(Oracle& f, bool total, Oracle& w, i64 w_max, i64 K, int64_t* h_spl_out) {
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  if (f.dev.kind == CPB_MODEL_BLOCK || f.dev.kind == CPB_MODEL_COLBLOCK)
    throw Error(CPB_ERR_UNSUPPORTED, "dynamic splitters need an affine random-access oracle");
  const Windows win = windows_weighted(w, w_max);
  oracle_ensure_ranks(f);
  if (f.dev.is_float) dynamic_constrained_T<double>(f, total, win, K, h_spl_out); else dynamic_constrained_T<i64>(f, total, win, K, h_spl_out);
}

// partition_stripe(A, K, ConvexTotalSplitter(f)) (ConvexTotalChunker.jl:26-55): the total-cost layers with the
// stack algorithm's tie rule.  Only for cost models that obey the quadrangle inequality the algorithm assumes
// (:121) -- work, connectivity and monotonized-symmetric models with non-negative coefficients; for anything else
// the reference's result is an artefact of its candidate stack and is not reproduced here.
void solve_convex_splitter(Oracle& f, const cpb_constraint* con, i64 K, int64_t* h_spl_out) {
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  bool convex = f.mdl.kind == CPB_MODEL_WORK || f.mdl.kind == CPB_MODEL_CONNECTIVITY || f.mdl.kind == CPB_MODEL_MONOSYM;
  for (int t = 1; t <= 3; ++t) convex = convex && f.mdl.coef[t] >= 0;
  if (!convex) throw Error(CPB_ERR_UNSUPPORTED, "ConvexTotalSplitter on the device needs a cost model obeying the quadrangle inequality (work / connectivity / monotonized-symmetric, beta >= 0)");
  if (con && con->enabled) {  // ConvexTotalChunker.jl:167-209
    const Windows win = windows_affine(*f.A, con);
    oracle_ensure_ranks(f);
    if (f.dev.is_float) convex_constrained_T<double>(f, win, K, h_spl_out); else convex_constrained_T<i64>(f, win, K, h_spl_out);
    return;
  }
  if (K == 1) {  // :33-35
    h_spl_out[0] = 1;
    h_spl_out[1] = f.A->n + 1;
    return;
  }
  oracle_ensure_ranks(f);
  if (f.dev.is_float) dynamic_T<double, TIE_CONVEX>(f, true, K, h_spl_out); else dynamic_T<i64, TIE_CONVEX>(f, true, K, h_spl_out);
}

// ConvexTotalSplitter(ConstrainedCost(f, w, w_max)) with a count weight w
void solve_convex_weighted(Oracle& f, Oracle& w, i64 w_max, i64 K, int64_t* h_spl_out) {
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  bool convex = f.mdl.kind == CPB_MODEL_WORK || f.mdl.kind == CPB_MODEL_CONNECTIVITY || f.mdl.kind == CPB_MODEL_MONOSYM;
  for (int t = 1; t <= 3; ++t) convex = convex && f.mdl.coef[t] >= 0;
  if (!convex) throw Error(CPB_ERR_UNSUPPORTED, "ConvexTotalSplitter on the device needs a cost model obeying the quadrangle inequality (work / connectivity / monotonized-symmetric, beta >= 0)");
  const Windows win = windows_weighted(w, w_max);
  oracle_ensure_ranks(f);
  if (f.dev.is_float) convex_constrained_T<double>(f, win, K, h_spl_out); else convex_constrained_T<i64>(f, win, K, h_spl_out);
}

}  // namespace cpb
