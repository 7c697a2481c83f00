// chunk.cu -- pack_stripe: the VBR chunkers.
//
//   DynamicTotalChunker   DynamicChunker.jl:20-75      windowed 1-D DP, ties -> smallest j
//   ConvexTotalChunker    ConvexTotalChunker.jl:141-265 same optimum; pointer rule of SURVEY App. B
//   OverlapChunker        OverlapChunker.jl:6-75       greedy on |rows(j) /\ rows(j')|
//   StrictChunker         StrictChunker.jl:5-54        greedy on identical column patterns
//   EquiChunker           EquiPartitioner.jl:15-21
//
// Kernel families:
//   window_cost_table  c(j'-t, j') for t = 1..W as a streaming pass: the stateful step oracles of the
//                      reference (SparseStepwiseDominanceCount, BlockComponentCostStepOracle
//                      BlockCosts.jl:68-142) become per-column suffix histograms of the link distance
//                      c - prev, summed along anti-diagonals.
//   chunk_dp_window    the chain cst[j'] = min_t cst[j'-t] + c(j'-t, j') is a (min,+) matrix product
//                      chain over W-vectors: blocks of columns compute their W x W transfer matrix in
//                      parallel, one warp combines them, blocks replay with their true entry state.
//                      Integer costs make re-association exact.
//   chain unravel      the pointer chain (bounded jumps) is marked block-wise the same way and
//                      compacted with a scan.
#include <algorithm>
#include <type_traits>
#include "engine.cuh"
#include "primitives.cuh"

namespace cpb {

static constexpr i64 CH_INF = (i64)1 << 60;
static constexpr int CH_BLOCK = 1024;  // columns per DP block
static constexpr int CH_MAXW = 64;     // widest supported window

static unsigned grid_for(size_t n) { return (unsigned)std::max<size_t>(1, std::min<size_t>((n + 255) / 256, (size_t)ctx().sm_count * 32)); }
static unsigned grid_t(size_t n, int threads) { return (unsigned)std::max<size_t>(1, (n + threads - 1) / threads); }

// ------------------------------------------------------------------------------------------------
// window_cost_table
// ------------------------------------------------------------------------------------------------

// G[r][(c-1)*W + (s-1)] = sum of weights of the points of column c whose link distance c - prev is >= s
// (s = 1..W).  One thread per column; the W suffix sums live in registers (WM = W rounded up to 8/16/32/64).
// wgt == nullptr: unit weights (plain distinct-row counting).
template <int WM>
__global__ void __launch_bounds__(128) k_window_hist(const u32* __restrict__ pos, const u32* __restrict__ ids, const u32* __restrict__ prev, u32 n, int W, int R,
                                                      const i64* __restrict__ wgt /* [R][nids] or null */, u32 nids, i64* __restrict__ G) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t c0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; c0 < n; c0 += stride) {
    const u32 c = (u32)c0 + 1;
    const u32 q0 = pos[c0], q1 = pos[c0 + 1];
    for (int r = 0; r < R; ++r) {
      i64 h[WM];
#pragma unroll
      for (int s = 0; s < WM; ++s) h[s] = 0;
      for (u32 q = q0; q < q1; ++q) {
        const u32 d = c - prev[q];
        const i64 w = wgt ? wgt[(size_t)r * nids + ids[q]] : 1;
#pragma unroll
        for (int s = 0; s < WM; ++s) h[s] += (d > (u32)s) ? w : 0;  // distance >= s + 1
      }
      i64* out = G + ((size_t)r * n + c0) * W;
#pragma unroll
      for (int s = 0; s < WM; ++s)
        if (s < W) out[s] = h[s];
    }
  }
}
static void window_hist(const u32* pos, const u32* ids, const u32* prev, u32 n, int W, int R, const i64* wgt, u32 nids, i64* G) {
  const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>(((size_t)n + 127) / 128, (size_t)ctx().sm_count * 64));
  if (W <= 8) CPB_LAUNCH(k_window_hist<8>, grid, 128, 0, pos, ids, prev, n, W, R, wgt, nids, G);
  else if (W <= 16) CPB_LAUNCH(k_window_hist<16>, grid, 128, 0, pos, ids, prev, n, W, R, wgt, nids, G);
  else if (W <= 32) CPB_LAUNCH(k_window_hist<32>, grid, 128, 0, pos, ids, prev, n, W, R, wgt, nids, G);
  else CPB_LAUNCH(k_window_hist<64>, grid, 128, 0, pos, ids, prev, n, W, R, wgt, nids, G);
}

struct TableModel {
  int kind, R, W;
  i64 a, bv, bp, bn;       // affine coefficients (Int64)
  double fa, fbv, fbp, fbn;
  const i64* alpha_col;    // [W+1]  (COLBLOCK / BLOCK)
  const i64* beta_col;     // [R][W+1]
  i64 wa, wbv, wbp, w_max; // weight constraint
};

// C[(jp-1)*W + (t-1)] = cost of the part [jp-t, jp), CH_INF if it violates the constraint or jp-t < 1
template <class T>
__global__ void k_cost_table(const u32* __restrict__ pos, u32 n, TableModel m, const i64* __restrict__ G, T* __restrict__ C, T inf) {
  const size_t total = ((size_t)n + 1) * m.W;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
    const u32 jp = (u32)(idx / m.W) + 1;
    const int t = (int)(idx % m.W) + 1;
    T c = inf;
    if ((i64)jp - t >= 1) {
      const u32 j = jp - t;
      const i64 np = (i64)pos[jp - 1] - (i64)pos[j - 1];
      if (m.wa + (i64)t * m.wbv + np * m.wbp <= m.w_max) {
        i64 d[4] = {0, 0, 0, 0};
        if (m.kind != CPB_MODEL_WORK)
          for (int r = 0; r < m.R; ++r)
            for (int i = 0; i < t; ++i) d[r] += G[((size_t)r * n + (j - 1 + i)) * m.W + i];
        constexpr bool IS_INT = (T)0.5 == (T)0;  // Int64 vs Float64 cost type
        if (m.kind == CPB_MODEL_WORK) {
          if (IS_INT) c = (T)(m.a + (i64)t * m.bv + np * m.bp);
          else c = (T)(m.fa + (double)t * m.fbv + (double)np * m.fbp);
        } else if (m.kind == CPB_MODEL_CONNECTIVITY) {
          if (IS_INT) c = (T)(m.a + (i64)t * m.bv + np * m.bp + d[0] * m.bn);
          else c = (T)(m.fa + (double)t * m.fbv + (double)np * m.fbp + (double)d[0] * m.fbn);
        } else if (m.kind == CPB_MODEL_COLBLOCK) {
          c = (T)(m.alpha_col[t] + d[0] * m.beta_col[t]);
        } else {  // BLOCK: alpha_col(w) + sum_r d_r * beta_col[r](w)   (BlockCosts.jl:132-136)
          i64 acc = m.alpha_col[t];
          for (int r = 0; r < m.R; ++r) acc += d[r] * m.beta_col[(size_t)r * (m.W + 1) + t];
          c = (T)acc;
        }
      }
    }
    C[idx] = c;
  }
}

// ------------------------------------------------------------------------------------------------
// chunk_dp_window (Int64 costs): blocked (min,+) scan
// ------------------------------------------------------------------------------------------------

// state x[t] = cst[jb - t], t = 0..W-1, for the boundary jb in front of the block
template <int WM>
__device__ __forceinline__ void dp_block_run(const i64* __restrict__ C, int W, u32 jp_first, u32 jp_last, i64 (&x)[WM], i64* __restrict__ cst,
                                             u32* __restrict__ ptr) {
  for (u32 jp = jp_first; jp <= jp_last; ++jp) {
    const i64* row = C + (size_t)(jp - 1) * W;
    i64 best = CH_INF;
    int bt = 0;
#pragma unroll
    for (int t = WM; t >= 1; --t) {  // descending t = ascending j: strict `<` keeps the smallest j (DynamicChunker.jl:45)
      if (t <= W) {
        const i64 c = x[t - 1] + row[t - 1];
        if (c < best) { best = c; bt = t; }
      }
    }
    if (best >= CH_INF) { best = CH_INF; bt = 0; }
#pragma unroll
    for (int t = WM - 1; t >= 1; --t) x[t] = x[t - 1];
    x[0] = best;
    if (cst) cst[jp] = best;
    if (ptr) ptr[jp] = bt ? jp - bt : 0;
  }
}

// M[b][i][t]: end state of block b when started from the unit state e_i
template <int WM>
__global__ void __launch_bounds__(128) k_chunk_transfer(const i64* __restrict__ C, u32 n, int W, u32 nblocks, i64* __restrict__ M) {
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= (size_t)nblocks * W) return;
  const u32 b = (u32)(tid / W);
  const int i = (int)(tid % W);
  i64 x[WM];
#pragma unroll
  for (int t = 0; t < WM; ++t) x[t] = (t == i) ? 0 : CH_INF;
  const u32 jb = 1 + b * CH_BLOCK;  // boundary in front of the block
  const u32 last = min(jb + CH_BLOCK, n + 1);
  dp_block_run<WM>(C, W, jb + 1, last, x, nullptr, nullptr);
  i64* out = M + ((size_t)b * W + i) * W;
#pragma unroll
  for (int t = 0; t < WM; ++t)
    if (t < W) out[t] = x[t];
}

// one warp walks the blocks: S[b][t] = true entry state of block b
__global__ void k_chunk_combine(const i64* __restrict__ M, u32 nblocks, int W, i64* __restrict__ S) {
  __shared__ i64 x[CH_MAXW];
  const int t = threadIdx.x;
  if (t < W) x[t] = (t == 0) ? 0 : CH_INF;  // cst[1] = 0, nothing before column 1
  __syncthreads();
  for (u32 b = 0; b < nblocks; ++b) {
    if (t < W) S[(size_t)b * W + t] = x[t];
    i64 y = CH_INF;
    if (t < W) {
      const i64* Mb = M + (size_t)b * W * W;
      for (int i = 0; i < W; ++i) {
        const i64 v = x[i] + Mb[(size_t)i * W + t];
        y = min(y, v);
      }
      if (y >= CH_INF) y = CH_INF;
    }
    __syncthreads();
    if (t < W) x[t] = y;
    __syncthreads();
  }
}

template <int WM>
__global__ void __launch_bounds__(128) k_chunk_final(const i64* __restrict__ C, u32 n, int W, u32 nblocks, const i64* __restrict__ S,
                                                     i64* __restrict__ cst, u32* __restrict__ ptr) {
  const u32 b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nblocks) return;
  i64 x[WM];
#pragma unroll
  for (int t = 0; t < WM; ++t) x[t] = (t < W) ? S[(size_t)b * W + t] : CH_INF;
  const u32 jb = 1 + b * CH_BLOCK;
  const u32 last = min(jb + CH_BLOCK, n + 1);
  if (b == 0) { cst[1] = 0; ptr[1] = 0; }
  dp_block_run<WM>(C, W, jb + 1, last, x, cst, ptr);
}


// ---- warp-per-block forms (W <= 32) -------------------------------------------------------------------------------
// The thread-per-block kernels above wait a full memory latency per DP step (ncu: k_chunk_final 1.5 ms, k_chunk_combine
// 4.3 ms at n = 4M).  Here a warp owns a block: the cost rows are fetched 256 values at a time with coalesced loads, one
// batch ahead of the chain, and staged in shared memory; lane i < W runs the chain started from the unit state e_i
// (transfer) or every lane runs the true state (final, lane 0 writes).
static constexpr int CW_WARPS = 8;
template <int WM, bool FINAL>
__global__ void __launch_bounds__(32 * CW_WARPS) k_chunk_warp(const i64* __restrict__ C, u32 n, int W, u32 nblocks, const i64* __restrict__ S,
                                                             i64* __restrict__ M, i64* __restrict__ cst, u32* __restrict__ ptr) {
  __shared__ i64 s_rows[CW_WARPS][2][256];
  const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
  const u32 b = blockIdx.x * CW_WARPS + wi;
  if (b >= nblocks) return;  // warp-uniform; only __syncwarp below
  const int RB = 256 / W;    // rows per batch (>= 8 for W <= 32)
  const u32 jb = 1 + b * CH_BLOCK;
  const u32 first = jb + 1, last = min(jb + CH_BLOCK, n + 1);
  i64 x[WM];
#pragma unroll
  for (int t = 0; t < WM; ++t) x[t] = FINAL ? (t < W ? S[(size_t)b * W + t] : CH_INF) : ((t == lane) ? 0 : CH_INF);
  if (FINAL && b == 0 && lane == 0) { cst[1] = 0; ptr[1] = 0; }
  i64 pre[8];
  auto fetch = [&](u32 jp0) {  // rows jp0 .. jp0 + RB - 1 (clipped to the block) -> registers
    const size_t base = (size_t)(jp0 - 1) * W;
    const u32 total = (u32)min((u32)RB, last - jp0 + 1) * (u32)W;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const u32 idx = (u32)k * 32 + lane;
      pre[k] = idx < total ? C[base + idx] : CH_INF;
    }
  };
  auto stash = [&](int slot) {
#pragma unroll
    for (int k = 0; k < 8; ++k) s_rows[wi][slot][k * 32 + lane] = pre[k];
  };
  if (first <= last) {
    fetch(first);
    stash(0);
  }
  __syncwarp();
  int slot = 0;
  for (u32 jp0 = first; jp0 <= last; jp0 += RB, slot ^= 1) {
    const bool more = (u64)jp0 + RB <= last;
    if (more) fetch(jp0 + RB);  // in flight while the chain below runs
    const u32 cnt = min((u32)RB, last - jp0 + 1);
#pragma unroll 4
    for (u32 r = 0; r < cnt; ++r) {
      const i64* row = &s_rows[wi][slot][r * W];
      // candidates t = W .. 2 only use states that are at least one step old: their minimum is off the critical path;
      // the chain itself is  best = (x[0] + row[0] < rest) ? x[0] + row[0] : rest.
      // descending t = ascending j: strict `<` keeps the smallest j (DynamicChunker.jl:45)
      i64 rest = CH_INF;
      int rt = 0;
#pragma unroll
      for (int t = WM; t >= 2; --t) {
        if (t <= W) {
          const i64 c = x[t - 1] + row[t - 1];
          if (c < rest) { rest = c; rt = t; }
        }
      }
      const i64 c1 = x[0] + row[0];
      i64 best = rest;
      int bt = rt;
      if (c1 < rest) { best = c1; bt = 1; }
      if (best >= CH_INF) { best = CH_INF; bt = 0; }
#pragma unroll
      for (int t = WM - 1; t >= 1; --t) x[t] = x[t - 1];
      x[0] = best;
      if (FINAL && lane == 0) {
        const u32 jp = jp0 + r;
        cst[jp] = best;
        ptr[jp] = bt ? jp - bt : 0;
      }
    }
    __syncwarp();  // everyone is done with s_rows[slot ^ 1]'s previous contents (read one iteration ago)
    if (more) stash(slot ^ 1);
    __syncwarp();
  }
  if (!FINAL && lane < W) {
    i64* out = M + ((size_t)b * W + lane) * W;
#pragma unroll
    for (int t = 0; t < WM; ++t)
      if (t < W) out[t] = x[t];
  }
}

// One warp walks the blocks with the state in registers (lane t holds x[t]).  The whole CTA stages the transfer
// matrices of CB_CHUNK blocks at a time in shared memory (coalesced), one chunk ahead of the walking warp, so a step
// costs a few shuffles instead of a memory latency (a one-block look-ahead in registers still paid ~0.5 us per block).
static constexpr int CB_THREADS = 256;
template <int WM>
__global__ void __launch_bounds__(CB_THREADS) k_chunk_combine_warp(const i64* __restrict__ M, u32 nblocks, int W, i64* __restrict__ S) {
  constexpr int CHUNK_VALS = 2560;  // i64 values per staged chunk (20 KB), two buffers
  __shared__ i64 s_m[2][CHUNK_VALS];
  const int tid = threadIdx.x;
  const u32 per = (u32)W * (u32)W;
  const u32 cb = max(1u, (u32)CHUNK_VALS / per);  // blocks per chunk
  const size_t total = (size_t)nblocks * per;
  auto stage = [&](u32 chunk, int buf, int first_thread) {  // by threads first_thread .. CB_THREADS - 1
    const size_t base = (size_t)chunk * cb * per;
    const u32 cnt = (u32)min((size_t)cb * per, total > base ? total - base : (size_t)0);
    for (u32 i = tid - first_thread; i < cnt; i += CB_THREADS - first_thread) s_m[buf][i] = M[base + i];
  };
  const u32 nchunks = (nblocks + cb - 1) / cb;
  if (nchunks) stage(0, 0, 0);
  __syncthreads();
  i64 x = (tid == 0) ? 0 : CH_INF;  // cst[1] = 0, nothing before column 1   (warp 0, lane t holds x[t])
  for (u32 ch = 0; ch < nchunks; ++ch) {
    const int buf = ch & 1;
    if (tid >= 32) {
      if (ch + 1 < nchunks) stage(ch + 1, buf ^ 1, 32);  // warps 1.. prefetch the next chunk
    } else {
      const u32 b0 = ch * cb, b1 = min(nblocks, b0 + cb);
      for (u32 b = b0; b < b1; ++b) {
        const i64* Mb = &s_m[buf][(size_t)(b - b0) * per];
        if (tid < W) S[(size_t)b * W + tid] = x;
        i64 cand[WM];
#pragma unroll
        for (int i = 0; i < WM; ++i) {
          const i64 xi = __shfl_sync(0xffffffffu, x, i);
          cand[i] = (i < W && tid < W) ? xi + Mb[i * W + tid] : CH_INF;
        }
#pragma unroll
        for (int span = WM / 2; span >= 1; span >>= 1)  // tree minimum: depth log2(WM) instead of WM
#pragma unroll
          for (int i = 0; i < span; ++i) cand[i] = min(cand[i], cand[i + span]);
        x = cand[0] >= CH_INF ? CH_INF : cand[0];
      }
    }
    __syncthreads();
  }
}

// Float64 costs: re-association would change roundings, so the chain runs in order on one thread
__global__ void k_chunk_seq_f64(const double* __restrict__ C, u32 n, int W, double* __restrict__ cst, u32* __restrict__ ptr) {
  if (blockIdx.x || threadIdx.x) return;
  cst[1] = 0.0;
  ptr[1] = 0;
  for (u32 jp = 2; jp <= n + 1; ++jp) {
    const double* row = C + (size_t)(jp - 1) * W;
    double best = INFINITY;
    int bt = 0;
    for (int t = min((u32)W, jp - 1); t >= 1; --t) {
      const double c = cst[jp - t] + row[t - 1];
      if (c < best) { best = c; bt = t; }
    }
    cst[jp] = best;
    ptr[jp] = bt ? jp - bt : 0;
  }
}

// ConvexTotalChunker{ConstrainedCost} pointer rule (SURVEY App. B; ConvexTotalChunker.jl:211-265):
// windows B_t = (b_t, b_t+1]; within the current window the leftmost argmin, unless the
// previous window is strictly better -- then its rightmost argmin.  The window ends b_t come from
// k_convex_bounds (bnd, nb of them); bnd == nullptr: a vertex-count weight, b_t = 1 + t W.
template <class T>
__global__ void k_convex_ptr(const T* __restrict__ C, const T* __restrict__ cst, u32 n, int W, const u32* __restrict__ bnd, const u32* __restrict__ nb,
                             u32* __restrict__ ptr) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const u32 jp = (u32)i + 2;
    u32 j0 = 1 + ((jp - 2) / W) * W;
    if (bnd) {  // the last window end before jp (bnd[0] = 1 < jp)
      u32 lo = 0, hi = *nb - 1;
      while (lo < hi) {
        const u32 mid = (lo + hi + 1) >> 1;
        if (bnd[mid] < jp) lo = mid; else hi = mid - 1;
      }
      j0 = bnd[lo];
    }
    const T* row = C + (size_t)(jp - 1) * W;
    bool has_in = false, has_pr = false;
    T vin = 0, vpr = 0;
    u32 ain = 0, apr = 0;
    for (int t = min((u32)W, jp - 1); t >= 1; --t) {  // ascending j
      const u32 j = jp - t;
      const T c = cst[j] + row[t - 1];
      if (j >= j0) {
        if (!has_in || c < vin) { vin = c; ain = j; has_in = true; }    // leftmost
      } else {
        if (!has_pr || c <= vpr) { vpr = c; apr = j; has_pr = true; }   // rightmost
      }
    }
    ptr[jp] = (!has_pr || (has_in && vin <= vpr)) ? ain : apr;
  }
}

// Window ends of a pin-weighted constraint: the reference moves from window to window by the weight's reach
// (ConvexTotalChunker.jl:211-265) -- b_0 = 1, b_t+1 = the last j' with w(b_t, j') <= w_max (at least b_t + 1) -- and a pin
// term makes that reach depend on the column lengths.  One thread walks the chain with binary searches on pos.
__global__ void k_convex_bounds(const u32* __restrict__ pos, u32 n, int W, i64 wa, i64 wbv, i64 wbp, i64 w_max, u32* __restrict__ bnd,
                                u32* __restrict__ nb) {
  if (blockIdx.x || threadIdx.x) return;
  u32 b = 1, k = 0;
  bnd[k++] = 1;
  while (b < n + 1) {
    u32 lo = b + 1, hi = min(b + (u32)W, n + 1);
    while (lo < hi) {
      const u32 mid = (lo + hi + 1) >> 1;
      if (wa + (i64)(mid - b) * wbv + ((i64)pos[mid - 1] - (i64)pos[b - 1]) * wbp <= w_max) lo = mid; else hi = mid - 1;
    }
    b = lo;
    bnd[k++] = b;
  }
  *nb = k;
}

// ------------------------------------------------------------------------------------------------
// chain unravel: nodes 1..n+1, forward pointers nxt[u] in (u, u + W], the chain runs 1 -> n+1
// ------------------------------------------------------------------------------------------------
static constexpr int UN_BLOCK = 512;

// DIR = +1: nxt is used as is.  DIR = -1: the chain is given by backward pointers ptr[j'] < j' and is
// walked in mirrored coordinates u = n + 2 - j'.
template <int DIR> __device__ __forceinline__ u32 chain_next(const u32* __restrict__ p, u32 u, u32 n) {
  if (DIR > 0) return p[u];
  return n + 2 - p[n + 2 - u];
}

template <int DIR>
__global__ void k_chain_exits(const u32* __restrict__ p, u32 n, int W, u32 nblocks, u32* __restrict__ exits) {
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= (size_t)nblocks * W) return;
  const u32 b = (u32)(tid / W), e = (u32)(tid % W);
  const u32 lo = 1 + b * UN_BLOCK, hi = min(lo + UN_BLOCK - 1, n + 1);  // nodes of the block
  u32 u = lo + e;
  while (u <= hi && u < n + 1) u = chain_next<DIR>(p, u, n);
  exits[tid] = (u > hi) ? u - (hi + 1) : 0xffffffffu;  // offset into the next block, or "ended here"
}

__global__ void k_chain_entries(const u32* __restrict__ exits, int W, u32 nblocks, u32* __restrict__ entry) {
  if (blockIdx.x || threadIdx.x) return;
  u32 e = 0;
  for (u32 b = 0; b < nblocks; ++b) {
    entry[b] = e;
    if (e == 0xffffffffu) continue;
    e = exits[(size_t)b * W + e];
  }
}

// The whole CTA stages the exit tables of many blocks in shared memory, one chunk ahead; thread 0 then resolves a block
// with one shared-memory read instead of one dependent global read.
static constexpr int CE_THREADS = 256;
__global__ void __launch_bounds__(CE_THREADS) k_chain_entries_staged(const u32* __restrict__ exits, int W, u32 nblocks, u32* __restrict__ entry) {
  constexpr int CHUNK_VALS = 5120;  // 20 KB per buffer
  __shared__ u32 s_e[2][CHUNK_VALS];
  const int tid = threadIdx.x;
  const u32 cb = max(1u, (u32)CHUNK_VALS / (u32)W);
  const size_t total = (size_t)nblocks * W;
  auto stage = [&](u32 chunk, int buf, int first_thread) {  // by threads first_thread .. CE_THREADS - 1
    const size_t base = (size_t)chunk * cb * W;
    const u32 cnt = (u32)min((size_t)cb * W, total > base ? total - base : (size_t)0);
    for (u32 i = tid - first_thread; i < cnt; i += CE_THREADS - first_thread) s_e[buf][i] = exits[base + i];
  };
  const u32 nchunks = (nblocks + cb - 1) / cb;
  if (nchunks) stage(0, 0, 0);
  __syncthreads();
  u32 e = 0;
  for (u32 ch = 0; ch < nchunks; ++ch) {
    const int buf = ch & 1;
    if (tid != 0) {
      if (ch + 1 < nchunks) stage(ch + 1, buf ^ 1, 1);
    } else {
      const u32 b0 = ch * cb, b1 = min(nblocks, b0 + cb);
      for (u32 b = b0; b < b1; ++b) {
        entry[b] = e;
        if (e != 0xffffffffu) e = s_e[buf][(size_t)(b - b0) * W + e];
      }
    }
    __syncthreads();
  }
}

template <int DIR>
__global__ void k_chain_mark(const u32* __restrict__ p, u32 n, u32 nblocks, const u32* __restrict__ entry, u32* __restrict__ flags) {
  const u32 b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nblocks || entry[b] == 0xffffffffu) return;
  const u32 lo = 1 + b * UN_BLOCK, hi = min(lo + UN_BLOCK - 1, n + 1);
  u32 u = lo + entry[b];
  while (u <= hi) {
    flags[u] = 1;
    if (u >= n + 1) break;
    u = chain_next<DIR>(p, u, n);
  }
}

template <int DIR>
__global__ void k_chain_emit(const u32* __restrict__ flags, const u32* __restrict__ scan, u32 n, u32 total, i64* __restrict__ spl) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x + 1; u <= (size_t)n + 1; u += stride)
    if (flags[u]) {
      if (DIR > 0) spl[scan[u]] = (i64)u;
      else spl[total - 1 - scan[u]] = (i64)(n + 2 - u);
    }
}

// -> host split vector; returns K
template <int DIR> static i64 unravel_chain(const u32* p, u32 n, int W, int64_t* h_spl_out) {
  const u32 nblocks = (u32)(((size_t)n + 1 + UN_BLOCK - 1) / UN_BLOCK);
  DBuf<u32> exits((size_t)nblocks * W), entry(nblocks), flags((size_t)n + 3), scan((size_t)n + 3);
  flags.zero();
  CPB_LAUNCH(k_chain_exits<DIR>, grid_t((size_t)nblocks * W, 128), 128, 0, p, n, W, nblocks, exits.get());
  CPB_LAUNCH(k_chain_entries_staged, 1, CE_THREADS, 0, exits.get(), W, nblocks, entry.get());
  CPB_LAUNCH(k_chain_mark<DIR>, grid_t(nblocks, 128), 128, 0, p, n, nblocks, entry.get(), flags.get());
  exclusive_scan_u32(flags.get(), scan.get(), (size_t)n + 3);
  u32 total = 0;
  CPB_CUDA(cudaMemcpyAsync(&total, scan.get() + n + 2, sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  CPB_REQUIRE(total >= 1, "empty chain");
  DBuf<i64> spl(total);
  CPB_LAUNCH(k_chain_emit<DIR>, grid_for((size_t)n + 1), 256, 0, flags.get(), scan.get(), n, total, spl.get());
  CPB_CUDA(cudaMemcpyAsync(h_spl_out, spl.get(), (size_t)total * sizeof(i64), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  return (i64)total - 1;
}

// ------------------------------------------------------------------------------------------------
// OverlapChunker / StrictChunker: independent next-boundary tables + chain unravel
// ------------------------------------------------------------------------------------------------

// nxt[j] = boundary after a chunk starting at column j (OverlapChunker.jl:37-67; note :29 -- the
// "cardinality of the first column" c is frozen at deg(column 1), SURVEY App. C)
__global__ void k_overlap_next(const u32* __restrict__ pos, const u32* __restrict__ row, u32 n, double rho, u32 w_max, u32* __restrict__ nxt) {
  const u32 c0 = pos[1] - pos[0];
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const u32 j = (u32)i + 1;
    u32 res = n + 1;
    for (u32 jp = j + 1; jp <= n; ++jp) {
      const u32 c2 = pos[jp] - pos[jp - 1];
      u32 cc = 0;  // |rows(j) /\ rows(jp)| by merging the two sorted lists
      u32 a = pos[j - 1], ae = pos[j], b = pos[jp - 1], be = pos[jp];
      while (a < ae && b < be) {
        const u32 ra = row[a], rb = row[b];
        cc += ra == rb;
        a += ra <= rb;
        b += rb <= ra;
      }
      if (jp - j == w_max || (double)cc < rho * (double)min(c0, c2)) { res = jp; break; }
    }
    nxt[j] = res;
  }
}

// eq[j'] = column j' has the same pattern as column j'-1 (1-based, j' >= 2)
__global__ void k_strict_next(const u32* __restrict__ pos, const u32* __restrict__ row, u32 n, u32 w_max, u32* __restrict__ nxt) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const u32 j = (u32)i + 1;
    u32 res = n + 1;
    const u32 a0 = pos[j - 1], len = pos[j] - pos[j - 1];
    for (u32 jp = j + 1; jp <= n; ++jp) {  // StrictChunker.jl:24-47
      bool same = (pos[jp] - pos[jp - 1] == len) && (jp - j != w_max);
      if (same) {
        const u32 b0 = pos[jp - 1];
        for (u32 l = 0; l < len; ++l)
          if (row[a0 + l] != row[b0 + l]) { same = false; break; }
      }
      if (!same) { res = jp; break; }
    }
    nxt[j] = res;
  }
}

// n_nets[k] = #distinct rows of chunk k (OverlapChunker.jl:61,69): rows of a column that do not occur
// in an earlier column of the same chunk, by binary search in the (sorted) earlier columns
__global__ void k_chunk_nets(const u32* __restrict__ pos, const u32* __restrict__ row, const i64* __restrict__ spl, i64 K, i64* __restrict__ out) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < (size_t)K; k += stride) {
    const u32 j = (u32)spl[k], jp = (u32)spl[k + 1];
    i64 d = 0;
    for (u32 c = j; c < jp; ++c)
      for (u32 q = pos[c - 1]; q < pos[c]; ++q) {
        const u32 r = row[q];
        bool seen = false;
        for (u32 c2 = j; c2 < c && !seen; ++c2) {
          u32 lo = pos[c2 - 1], hi = pos[c2];
          while (lo < hi) {
            const u32 mid = lo + ((hi - lo) >> 1);
            if (row[mid] < r) lo = mid + 1; else hi = mid;
          }
          seen = lo < pos[c2] && row[lo] == r;
        }
        d += !seen;
      }
    out[k] = d;
  }
}

// ------------------------------------------------------------------------------------------------
// BLOCK model: the matrix collapsed to (row part x column), duplicates inside a column removed
// ------------------------------------------------------------------------------------------------
__global__ void k_collapse_flags(const u32* __restrict__ pos, const u32* __restrict__ row, const u32* __restrict__ colidx,
                                 const u32* __restrict__ asg, size_t N, u32* __restrict__ keep) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q <= N; q += stride) {
    u32 k = 0;
    if (q < N) k = (q == pos[colidx[q]] || asg[row[q]] != asg[row[q - 1]]) ? 1u : 0u;
    keep[q] = k;
  }
}
__global__ void k_collapse_emit(const u32* __restrict__ row, const u32* __restrict__ asg, const u32* __restrict__ keep,
                                const u32* __restrict__ scan, size_t N, u32* __restrict__ ids) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < N; q += stride)
    if (keep[q]) ids[scan[q]] = asg[row[q]];
}
__global__ void k_collapse_pos(const u32* __restrict__ pos, const u32* __restrict__ scan, u32 n, u32* __restrict__ pos2) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j <= n; j += stride) pos2[j] = scan[pos[j]];
}
__global__ void k_part_weights(const u32* __restrict__ size, u32 K, int R, const i64* __restrict__ beta_row, int U, i64* __restrict__ wgt) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < K; k += stride)
    for (int r = 0; r < R; ++r) wgt[(size_t)r * K + k] = beta_row[(size_t)r * U + min(size[k], (u32)(U - 1))];
}

// ------------------------------------------------------------------------------------------------
template <int WM> static void run_dp_blocks(const i64* C, u32 n, int W, i64* cst, u32* ptr) {
  const u32 nblocks = (u32)(((size_t)n + CH_BLOCK - 1) / CH_BLOCK);
  if (nblocks == 0) return;
  DBuf<i64> M((size_t)nblocks * W * W), S((size_t)nblocks * W);
  if (WM <= 32 && !std::getenv("CPB_CHUNK_THREAD_BLOCKS")) {
    const unsigned g = (nblocks + CW_WARPS - 1) / CW_WARPS;
    CPB_LAUNCH((k_chunk_warp<WM, false>), g, 32 * CW_WARPS, 0, C, n, W, nblocks, (const i64*)nullptr, M.get(), (i64*)nullptr, (u32*)nullptr);
    CPB_LAUNCH(k_chunk_combine_warp<WM>, 1, CB_THREADS, 0, M.get(), nblocks, W, S.get());
    CPB_LAUNCH((k_chunk_warp<WM, true>), g, 32 * CW_WARPS, 0, C, n, W, nblocks, S.get(), (i64*)nullptr, cst, ptr);
    return;
  }
  CPB_LAUNCH(k_chunk_transfer<WM>, grid_t((size_t)nblocks * W, 128), 128, 0, C, n, W, nblocks, M.get());
  CPB_LAUNCH(k_chunk_combine, 1, CH_MAXW, 0, M.get(), nblocks, W, S.get());
  CPB_LAUNCH(k_chunk_final<WM>, grid_t(nblocks, 128), 128, 0, C, n, W, nblocks, S.get(), cst, ptr);
}

static void pack_dynamic(Matrix& A, Oracle& f, int method, const cpb_constraint* con, int64_t* h_spl_out, int64_t* K_out) {
  const u32 n = (u32)A.n;
  const size_t N = (size_t)A.N;
  const cpb_model& mdl = f.mdl;
  CPB_REQUIRE(con && con->enabled, "the device chunk DP needs a width constraint ConstrainedCost(f, w, w_max) (unconstrained block-cost chunking is an O(n^2) chain: not built)");
  CPB_REQUIRE(con->w_coef[1] >= 1 && con->w_coef[2] >= 0 && con->w_coef[0] >= 0, "weight must grow with the vertex count (VertexCount or AffineWorkModel(0, b_v >= 1, b_p >= 0))");
  if (n == 0) { h_spl_out[0] = 1; *K_out = 0; return; }
  const i64 Wl = std::min<i64>(n, (con->w_max - con->w_coef[0]) / con->w_coef[1]);
  if (Wl < 1) throw Error(CPB_ERR_INFEASIBLE, "width constraint admits no non-empty chunk (reference: @assert j0 < j')");
  CPB_REQUIRE(Wl <= CH_MAXW, "window wider than 64 columns is not supported on the device");
  const int W = (int)Wl;
  const bool is_f = mdl.is_float != 0;
  CPB_REQUIRE(mdl.kind == CPB_MODEL_WORK || mdl.kind == CPB_MODEL_CONNECTIVITY || mdl.kind == CPB_MODEL_COLBLOCK || mdl.kind == CPB_MODEL_BLOCK,
              "pack_stripe on the device supports work, connectivity, column-block and block cost models");
  if (mdl.kind == CPB_MODEL_COLBLOCK || mdl.kind == CPB_MODEL_BLOCK) {
    CPB_REQUIRE(!is_f, "block cost models are supported with Int64 components (as in every reference use)");
    CPB_REQUIRE(mdl.w_tab >= W, "block component tables are shorter than the window");
  }

  // ---- window_cost_table ----
  trace_mark("checks");
  TableModel tm{};
  tm.kind = mdl.kind; tm.W = W; tm.R = 1;
  tm.fa = mdl.coef[0]; tm.fbv = mdl.coef[1]; tm.fbp = mdl.coef[2]; tm.fbn = mdl.coef[3];
  tm.a = (i64)mdl.coef[0]; tm.bv = (i64)mdl.coef[1]; tm.bp = (i64)mdl.coef[2]; tm.bn = (i64)mdl.coef[3];
  tm.wa = con->w_coef[0]; tm.wbv = con->w_coef[1]; tm.wbp = con->w_coef[2]; tm.w_max = con->w_max;
  DBuf<i64> G, tabs, wgt;
  {
    ProfScope prof("window_cost_table", (double)(N + n + 1) * 4.0 + (double)n * W * 8.0);
    if (mdl.kind == CPB_MODEL_CONNECTIVITY || mdl.kind == CPB_MODEL_COLBLOCK) {
      DBuf<u32> prev(N), colidx(N);
      compute_prev_links(A.pos.get(), A.row.get(), (u32)A.m, n, N, prev.get(), colidx.get());
      G.alloc((size_t)n * W);
      window_hist(A.pos.get(), A.row.get(), prev.get(), n, W, 1, (const i64*)nullptr, 0u, G.get());
    } else if (mdl.kind == CPB_MODEL_BLOCK) {
      const int R = mdl.R;
      tm.R = R;
      const u32 Kp = (u32)f.pi_K;
      DBuf<u32> colidx(N), keep(N + 1), scan(N + 1);
      expand_columns(A.pos.get(), n, colidx.get(), N);
      CPB_LAUNCH(k_collapse_flags, grid_for(N + 1), 256, 0, A.pos.get(), A.row.get(), colidx.get(), f.pi_asg.get(), N, keep.get());
      exclusive_scan_u32(keep.get(), scan.get(), N + 1);
      u32 N2 = 0;
      CPB_CUDA(cudaMemcpyAsync(&N2, scan.get() + N, sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));
      DBuf<u32> ids(N2), pos2((size_t)n + 1), prev(N2), colidx2(N2);
      if (N) CPB_LAUNCH(k_collapse_emit, grid_for(N), 256, 0, A.row.get(), f.pi_asg.get(), keep.get(), scan.get(), N, ids.get());
      CPB_LAUNCH(k_collapse_pos, grid_for((size_t)n + 1), 256, 0, A.pos.get(), scan.get(), n, pos2.get());
      trace_mark("collapse");
      compute_prev_links(pos2.get(), ids.get(), Kp, n, N2, prev.get(), colidx2.get());
      trace_mark("links");
      // per-part weights beta_row[r](u_k)
      const int U = mdl.u_tab + 1;
      std::vector<i64> hbr((size_t)R * U);
      for (size_t t = 0; t < hbr.size(); ++t) hbr[t] = (i64)f.h_beta_row[t];
      DBuf<i64> dbr(hbr.size());
      CPB_CUDA(cudaMemcpyAsync(dbr.get(), hbr.data(), hbr.size() * sizeof(i64), cudaMemcpyHostToDevice, ctx().stream));
      wgt.alloc((size_t)R * Kp);
      if (Kp) CPB_LAUNCH(k_part_weights, grid_for(Kp), 256, 0, f.pi_size.get(), Kp, R, dbr.get(), U, wgt.get());
      G.alloc((size_t)R * n * W);
      window_hist(pos2.get(), ids.get(), prev.get(), n, W, R, wgt.get(), Kp, G.get());
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));  // hbr goes out of scope
    }
    if (mdl.kind == CPB_MODEL_COLBLOCK || mdl.kind == CPB_MODEL_BLOCK) {
      // tables re-laid out for widths 0..W
      const int R = tm.R, Wt = mdl.w_tab + 1;
      std::vector<i64> h((size_t)(R + 1) * (W + 1));
      const double* ac = f.h_alpha_col.data();
      const double* bc = f.h_beta_col.data();
      for (int w = 0; w <= W; ++w) h[w] = (i64)ac[w];
      for (int r = 0; r < R; ++r)
        for (int w = 0; w <= W; ++w) h[(size_t)(r + 1) * (W + 1) + w] = (i64)bc[(size_t)r * Wt + w];
      tabs.alloc(h.size());
      CPB_CUDA(cudaMemcpyAsync(tabs.get(), h.data(), h.size() * sizeof(i64), cudaMemcpyHostToDevice, ctx().stream));
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));
      tm.alpha_col = tabs.get();
      tm.beta_col = tabs.get() + (W + 1);
    }
  }
  trace_mark("window_hist");
  const size_t cells = ((size_t)n + 1) * W;
  DBuf<u32> ptr((size_t)n + 3);
  auto convex_ptr = [&](const auto* C, const auto* cst) {
    using T = std::remove_const_t<std::remove_pointer_t<decltype(C)>>;
    DBuf<u32> bnd, nb;
    if (tm.wbp != 0) {  // pin-weighted windows: their ends follow the column lengths
      bnd.alloc((size_t)n + 2);
      nb.alloc(1);
      CPB_LAUNCH(k_convex_bounds, 1, 32, 0, A.pos.get(), n, W, tm.wa, tm.wbv, tm.wbp, tm.w_max, bnd.get(), nb.get());
    }
    CPB_LAUNCH(k_convex_ptr<T>, grid_for(n), 256, 0, C, cst, n, W, (const u32*)bnd.get(), (const u32*)nb.get(), ptr.get());
  };
  if (!is_f) {
    DBuf<i64> C(cells), cst((size_t)n + 2);
    {
      ProfScope prof("window_cost_table");
      CPB_LAUNCH(k_cost_table<i64>, grid_for(cells), 256, 0, A.pos.get(), n, tm, G.get(), C.get(), (i64)CH_INF);
    }
    trace_mark("cost_table");
    {
      ProfScope prof("chunk_dp_window", (double)cells * 8.0 + (double)(n + 1) * 12.0);
      if (W <= 8) run_dp_blocks<8>(C.get(), n, W, cst.get(), ptr.get());
      else if (W <= 16) run_dp_blocks<16>(C.get(), n, W, cst.get(), ptr.get());
      else if (W <= 32) run_dp_blocks<32>(C.get(), n, W, cst.get(), ptr.get());
      else run_dp_blocks<64>(C.get(), n, W, cst.get(), ptr.get());
      i64 last = 0;
      CPB_CUDA(cudaMemcpyAsync(&last, cst.get() + n + 1, sizeof(i64), cudaMemcpyDeviceToHost, ctx().stream));
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));
      if (last >= CH_INF) throw Error(CPB_ERR_INFEASIBLE, "width constraint cannot be met (reference: @assert j0 < j')");
      if (method == CPB_PACK_CONVEX_TOTAL) convex_ptr(C.get(), cst.get());
    }
  } else {
    DBuf<double> C(cells), cst((size_t)n + 2);
    {
      ProfScope prof("window_cost_table");
      CPB_LAUNCH(k_cost_table<double>, grid_for(cells), 256, 0, A.pos.get(), n, tm, G.get(), C.get(), (double)INFINITY);
    }
    ProfScope prof("chunk_dp_window", (double)cells * 8.0 + (double)(n + 1) * 12.0);
    CPB_LAUNCH(k_chunk_seq_f64, 1, 32, 0, C.get(), n, W, cst.get(), ptr.get());
    double last = 0;
    CPB_CUDA(cudaMemcpyAsync(&last, cst.get() + n + 1, sizeof(double), cudaMemcpyDeviceToHost, ctx().stream));
    CPB_CUDA(cudaStreamSynchronize(ctx().stream));
    if (!(last < INFINITY)) throw Error(CPB_ERR_INFEASIBLE, "width constraint cannot be met (reference: @assert j0 < j')");
    if (method == CPB_PACK_CONVEX_TOTAL) convex_ptr(C.get(), cst.get());
  }
  trace_mark("chunk_dp");
  ProfScope prof("unravel_chunks");
  *K_out = unravel_chain<-1>(ptr.get(), n, W, h_spl_out);
  trace_mark("unravel");
}

void solve_pack(Matrix& A, Oracle* f, int method, const cpb_constraint* con, double rho, i64 w_max, int64_t* h_spl_out,
                int64_t* K_out, int64_t* n_nets_out) {
  const i64 n = A.n;
  switch (method) {
    case CPB_PACK_EQUI: {  // EquiPartitioner.jl:15-21: [1:w:n; n+1]
      CPB_REQUIRE(w_max >= 1, "EquiChunker width must be >= 1");
      i64 K = 0;
      for (i64 j = 1; j <= n; j += w_max) h_spl_out[K++] = j;
      h_spl_out[K] = n + 1;
      *K_out = K;
      return;
    }
    case CPB_PACK_DYNAMIC_TOTAL:
    case CPB_PACK_CONVEX_TOTAL:
      CPB_REQUIRE(f != nullptr, "pack_stripe: this method needs a cost oracle");
      if (!(con && con->enabled) && f->mdl.kind != CPB_MODEL_BLOCK && f->mdl.kind != CPB_MODEL_COLBLOCK) {
        // pack_stripe(A, ConvexTotalChunker(f)) (ConvexTotalChunker.jl:9-24) and pack_stripe(A, DynamicTotalChunker(f))
        // (DynamicChunker.jl:15-56 with the FeasibleCost sentinel) without a width constraint.  For the affine
        // models that obey the quadrangle inequality the stack algorithm assumes (:121) -- work, connectivity,
        // monotonized-symmetric with alpha >= 0 and beta >= 0 -- costs are subadditive (f(1, j') <= f(1, j) + f(j, j') -
        // alpha), so j = 1 attains every minimum of cst[j'] = min_j cst[j] + f(j, j') and, being the smallest minimiser
        // (the rule chunk_convex! follows, SURVEY.md App. B, and the `<` of DynamicChunker.jl:45), is the pointer of every
        // j': the result is the single chunk [1, n + 1] (no chunk at all for n = 0) -- 2400/2400 and 1500/1500 random
        // cases against the restated algorithms in tests/test_oracle_solvers.py.  Nothing needs the device.
        const cpb_model& m = f->mdl;
        bool ok = m.kind == CPB_MODEL_WORK || m.kind == CPB_MODEL_CONNECTIVITY || m.kind == CPB_MODEL_MONOSYM;
        for (int t = 0; t <= 3; ++t) ok = ok && m.coef[t] >= 0;
        if (!ok)
          throw Error(CPB_ERR_UNSUPPORTED, "unconstrained Convex/DynamicTotalChunker needs a subadditive affine model with alpha, beta >= 0 "
                                           "(work / connectivity / monotonized-symmetric); anything else is an online least-weight-subsequence chain");
        h_spl_out[0] = 1;
        if (n >= 1) h_spl_out[1] = n + 1;
        *K_out = n >= 1 ? 1 : 0;
        return;
      }
      pack_dynamic(A, *f, method, con, h_spl_out, K_out);
      return;
    case CPB_PACK_OVERLAP:
    case CPB_PACK_STRICT: {
      CPB_REQUIRE(n >= 1, "chunker reads column 1: n >= 1 required");
      CPB_REQUIRE(w_max >= 1 && w_max <= CH_MAXW, "w_max must be in 1..64 on the device");
      ProfScope prof(method == CPB_PACK_OVERLAP ? "overlap_chunker" : "strict_chunker", (double)(A.N + n + 1) * 4.0);
      DBuf<u32> nxt((size_t)n + 3);
      if (method == CPB_PACK_OVERLAP)
        CPB_LAUNCH(k_overlap_next, grid_for((size_t)n), 256, 0, A.pos.get(), A.row.get(), (u32)n, rho, (u32)w_max, nxt.get());
      else
        CPB_LAUNCH(k_strict_next, grid_for((size_t)n), 256, 0, A.pos.get(), A.row.get(), (u32)n, (u32)w_max, nxt.get());
      const i64 K = unravel_chain<1>(nxt.get(), (u32)n, (int)w_max, h_spl_out);
      *K_out = K;
      if (method == CPB_PACK_OVERLAP && n_nets_out) {
        DBuf<i64> dspl(K + 1), dn(K);
        CPB_CUDA(cudaMemcpyAsync(dspl.get(), h_spl_out, (K + 1) * sizeof(i64), cudaMemcpyHostToDevice, ctx().stream));
        CPB_LAUNCH(k_chunk_nets, grid_for((size_t)K), 256, 0, A.pos.get(), A.row.get(), dspl.get(), K, dn.get());
        CPB_CUDA(cudaMemcpyAsync(n_nets_out, dn.get(), K * sizeof(i64), cudaMemcpyDeviceToHost, ctx().stream));
        CPB_CUDA(cudaStreamSynchronize(ctx().stream));
      }
      return;
    }
    case CPB_PACK_CONCAVE_TOTAL:  // ConcaveTotalChunker.jl:9-24 (concave.cu: the queue routine, one device thread)
      CPB_REQUIRE(f != nullptr, "pack_stripe: this method needs a cost oracle");
      solve_concave_chunker(*f, con, h_spl_out, K_out);
      return;
    default: throw Error(CPB_ERR_UNSUPPORTED, "unknown pack_stripe method");
  }
}

}  // namespace cpb
