// bisect.cu -- kernel family "probe": BisectCostBottleneckSplitter / LazyBisectCostBottleneckSplitter
// (BisectCostBottleneckSplitter.jl:6-63, LazyBisectCostBottleneckSplitter.jl:8-70,140-258,260-388).
//
// The reference bisects the cost value c = (c_lo + c_hi) / 2 and runs one greedy feasibility probe
// per threshold: part k extends as far right as c(spl[k], j', k) <= c allows.  The streaming
// ("lazy") and the random-access form return the same split vectors for monotone costs, so both
// map onto one engine here:
//   * the next `depth` levels of the bisection tree (2^depth - 1 thresholds, each computed with the
//     reference's own double expression) are probed CONCURRENTLY, one CTA per threshold, and the
//     tree is then walked by feasibility -- the threshold sequence, and therefore the returned
//     spl_hi, is identical to the sequential loop by construction;
//   * inside a probe, each part boundary is found by a multi-way search over a thread-block CLUSTER
//     (8 CTAs x 128 threads = 1024 candidates j' per round, every thread evaluates the oracle at one
//     candidate; counts are exchanged through distributed shared memory, one cluster barrier per
//     round) instead of the reference's one-query-at-a-time binary search.  Spreading a threshold
//     over 8 SMs matters: the rank descents are one random 32-byte sector per level and candidate,
//     and a single SM's L1 serialises them (ncu, profiles/r01).  Previous probes' windows
//     (spl_lo/spl_hi, BisectCost...:29-33,46,55,58) are used as search hints only; a miss falls
//     back to the full range, so the result never depends on them.
#include <algorithm>
#include <cmath>
#include <queue>
#include <cooperative_groups.h>
#include "engine.cuh"

namespace cg = cooperative_groups;

namespace cpb {

static constexpr int BS_THREADS = 128;
static constexpr int BS_CLUSTER = 8;
static constexpr int BS_WIDTH = BS_THREADS * BS_CLUSTER;  // candidates per round
static constexpr int BS_MAX_NODES = 255;    // nodes of one round's speculation tree (all ranks together)
static constexpr int BS_MAX_DEPTH = 24;     // deepest node of a round's tree (heap index < 2^25)
static constexpr int BS_LOCAL_DEPTH = 4;    // a single GPU hosts at most 2^4 clusters of 8 CTAs

struct BisectState {
  double c_lo, c_hi;
  int done;
  int probes;
  int rounds;
  int _pad;
};

// Threshold of the bisection-tree node with heap index `heap` (left child = "the parent's probe was feasible"),
// produced with the reference's own double expressions from the round's starting state; returns 0 if the
// sequential loop would have stopped before reaching the node.
__device__ __forceinline__ int node_threshold(const BisectState* __restrict__ st, double eps1, int heap, double* c_out) {
  int valid = (st->done || heap < 0) ? 0 : 1;  // heap < 0: unused slot of the round's plan
  double lo = st->c_lo, hi = st->c_hi;
  int len = 0;
  unsigned path = 0;  // bit t = step t (from the node upwards) was a left child
  for (int i = heap; i > 0; i = (i - 1) >> 1) { path |= (unsigned)(i & 1) << len; ++len; }
  for (int t = len - 1; t >= 0 && valid; --t) {
    if (!(lo * eps1 < hi)) { valid = 0; break; }
    const double c = (lo + hi) / 2;
    if ((path >> t) & 1u) hi = c; else lo = c;
  }
  if (valid && !(lo * eps1 < hi)) valid = 0;
  *c_out = (lo + hi) / 2;
  return valid;
}

// largest x in [a, b] with c(j, x) <= c, or a-1 if c(j, a) > c.  Monotone predicate.  Cluster-wide:
// every CTA of the cluster calls it with the same arguments and gets the same answer.
template <class T>
__device__ __forceinline__ i64 wide_search(const DevOracle& o, cg::cluster_group& cluster, int (*s_cnt)[BS_CLUSTER], int& phase,
                                           u32 j, i64 a, i64 b, double c, u32 k) {
  const unsigned crank = cluster.block_rank();
  while (true) {
    const i64 S = b - a + 1;
    if (S <= 0) return a - 1;
    const i64 stride = (S + BS_WIDTH - 1) / BS_WIDTH;
    const i64 x = a + (i64)(crank * BS_THREADS + threadIdx.x) * stride;
    bool ok = false;
    if (x <= b) ok = cost_leq(dev_cost<T>(o, j, (u32)x, k), c);
    const int mine = __syncthreads_count(ok);
    if (threadIdx.x < BS_CLUSTER) {  // push my count into slot [crank] of every CTA of the cluster
      int* remote = cluster.map_shared_rank(&s_cnt[phase][crank], threadIdx.x);
      *remote = mine;
    }
    cluster.sync();
    int ct = 0;
#pragma unroll
    for (int p = 0; p < BS_CLUSTER; ++p) ct += s_cnt[phase][p];
    phase ^= 1;  // double-buffered: a fast CTA may already be writing the next round's counts
    if (ct == 0) return a - 1;
    const i64 base = a + (i64)(ct - 1) * stride;
    if (stride == 1) return base;
    a = base + 1;
    b = min(b, base + stride - 1);
  }
}

template <class T>
__global__ void __cluster_dims__(BS_CLUSTER, 1, 1) __launch_bounds__(BS_THREADS)
    k_bisect_round(const __grid_constant__ DevOracle o, int K, double eps1, const BisectState* __restrict__ st,
                   const int* __restrict__ hint_lo, const int* __restrict__ hint_hi, int* __restrict__ node_spl,
                   int* __restrict__ node_res, double* __restrict__ node_c, const int* __restrict__ node_ids, int node_base) {
  __shared__ double s_c;
  __shared__ int s_valid;
  __shared__ int s_cnt[2][BS_CLUSTER];
  cg::cluster_group cluster = cg::this_cluster();
  const int node = node_base + blockIdx.x / BS_CLUSTER;  // slot of this round; node_ids[slot] = heap index in the bisection tree
  const bool writer = cluster.block_rank() == 0 && threadIdx.x == 0;
  if (threadIdx.x == 0) s_valid = node_threshold(st, eps1, node_ids[node], &s_c);
  __syncthreads();
  if (!s_valid) {  // uniform over the cluster: every CTA derives it from the same state
    if (writer) node_res[node] = 0;
    return;
  }
  const double c = s_c;
  const i64 n1 = (i64)o.n + 1;
  int* spl = node_spl + (size_t)node * (K + 2);  // 1-based, spl[1..K+1]
  if (writer) { spl[1] = 1; spl[K + 1] = (int)n1; }
  int phase = 0;
  i64 j = 1;
  bool broke = false;
  for (int k = 1; k <= K - 1; ++k) {
    i64 a = max(j, (i64)hint_lo[k + 1]);
    i64 b = min((i64)hint_hi[k + 1], n1);
    if (b < a) { a = j; b = n1; }
    i64 r = wide_search<T>(o, cluster, s_cnt, phase, (u32)j, a, b, c, (u32)k);
    if (r == a - 1 && a > j) r = wide_search<T>(o, cluster, s_cnt, phase, (u32)j, j, a - 1, c, (u32)k);
    else if (r == b && b < n1) r = wide_search<T>(o, cluster, s_cnt, phase, (u32)j, b + 1, n1, c, (u32)k);
    if (r < j) {  // even the empty part exceeds c (BisectCost...:47-51)
      broke = true;
      if (writer)
        for (int t = k + 1; t <= K; ++t) spl[t] = (int)j;
      break;
    }
    if (writer) spl[k + 1] = (int)r;
    j = r;
  }
  if (writer) {
    bool feas = false;
    if (!broke) feas = cost_leq(dev_cost<T>(o, (u32)j, (u32)n1, (u32)K), c);
    node_c[node] = c;
    node_res[node] = feas ? 2 : 1;
  }
  cluster.sync();  // no CTA may exit while peers can still write into its shared memory
}

// ------------------------------------------------------------------------------------------------
// BisectIndexBottleneckSplitter (BisectIndexBottleneckSplitter.jl:5-81): the EXACT bottleneck splitter.  Candidate
// thresholds are costs c(spl[k], j') of actual parts; for every part k a binary search over j' keeps the candidates
// inside [c_lo, c_hi) and tests each with a greedy probe of the remaining parts, searched inside the windows
// spl_lo / spl_hi left by earlier probes.  The whole control flow runs inside ONE kernel on one 8-CTA cluster (every
// thread follows the same deterministic sequence; the part searches are the 1024-way cluster searches of
// k_bisect_round), the windows are hard limits exactly as in the reference, so the split vector is the reference's.
// ------------------------------------------------------------------------------------------------
template <class T>
__device__ __forceinline__ void bisect_index_body(const DevOracle& o, int (*s_cnt)[BS_CLUSTER], int K, double c_lo, double c_hi, int* __restrict__ spl,
                                                  int* __restrict__ spl_lo, int* __restrict__ spl_hi, int* __restrict__ probes_out) {
  cg::cluster_group cluster = cg::this_cluster();
  const bool cta0 = cluster.block_rank() == 0;
  const bool writer = cta0 && threadIdx.x == 0;
  const i64 n1 = (i64)o.n + 1;
  if (cta0)
    for (int t = 1 + threadIdx.x; t <= K + 1; t += blockDim.x) {  // :29-37
      spl_lo[t] = (t == K + 1) ? (int)n1 : 1;
      spl_hi[t] = (t == 1) ? 1 : (int)n1;
      spl[t] = (t == 1) ? 1 : (t == K + 1 ? (int)n1 : 0);
    }
  __threadfence();
  cluster.sync();
  int phase = 0, probes = 0;
  i64 sk = 1;  // spl[k]
  for (int k = 1; k <= K; ++k) {
    i64 jp_hi = __ldcg(spl_hi + k + 1);
    i64 jp_lo = max(sk, (i64)__ldcg(spl_lo + k + 1));
    while (jp_lo <= jp_hi) {
      const i64 jp = (jp_lo + jp_hi) >> 1;
      const T c = dev_cost<T>(o, (u32)sk, (u32)jp, (u32)k);
      const double cd = (double)c;
      if (c_lo <= cd && cd < c_hi) {
        ++probes;
        bool chk = true;
        if (writer) spl[k + 1] = (int)jp;
        i64 j = jp;
        for (int kk = k + 1; kk <= K - 1; ++kk) {
          const i64 a = max(j, (i64)__ldcg(spl_lo + kk + 1));
          const i64 b = __ldcg(spl_hi + kk + 1);
          // search (:14-27): the largest j' in [a, b] with c(j, j') <= c; b if the window is empty, a - 1 if none fits
          const i64 r = a > b ? b : wide_search<T>(o, cluster, s_cnt, phase, (u32)j, a, b, cd, (u32)kk);
          if (writer) spl[kk + 1] = (int)r;
          if (r < j) {
            chk = false;
            if (cta0)
              for (int t = kk + 1 + threadIdx.x; t <= K; t += blockDim.x) spl[t] = (int)j;
            break;
          }
          j = r;
        }
        // the last part: [spl[K], spl[K+1])
        const i64 ls = (k == K) ? sk : j, le = (k == K) ? jp : n1;
        const bool feas = chk && cost_leq(dev_cost<T>(o, (u32)ls, (u32)le, (u32)K), cd);
        __syncthreads();  // CTA 0: the writer's spl entries are visible to the copying threads
        if (feas) { c_hi = cd; jp_hi = jp - 1; } else { c_lo = cd; jp_lo = jp + 1; }
        if (cta0) {
          int* dst = feas ? spl_hi : spl_lo;
          for (int t = 1 + threadIdx.x; t <= K + 1; t += blockDim.x) dst[t] = spl[t];
          __threadfence();
        }
        cluster.sync();  // the new window is visible to every CTA before the next search reads it
      } else if (cd >= c_hi) {
        jp_hi = jp - 1;
      } else {
        jp_lo = jp + 1;
      }
    }
    if (jp_hi < sk) break;
    if (writer) spl[k + 1] = (int)jp_hi;
    sk = jp_hi;
  }
  if (writer) *probes_out = probes;
  cluster.sync();  // no CTA may exit while peers can still write into its shared memory
}

// ------------------------------------------------------------------------------------------------
// The Flip family (costs that DEcrease as the part grows -- the secondary models): FlipBisectCostBottleneckSplitter
// (BisectCostBottleneckSplitter.jl:70-127), LazyFlipBisectCostBottleneckSplitter (LazyBisect...:79-138) and
// FlipBisectIndexBottleneckSplitter (BisectIndex...:87-166).  Each part is made as SHORT as the threshold allows.  These
// run as one kernel on one cluster that follows the reference's sequential control flow (hard windows included), with
// the 1024-way cluster search for "the smallest j' whose cost is <= c".
// ------------------------------------------------------------------------------------------------
// smallest x in [a, b] with c(j, x, k) <= c, b + 1 if none; a if the window is empty (the reference returns j'_lo).
// The predicate is monotone (false ... false true ... true).
template <class T>
__device__ __forceinline__ i64 wide_search_flip(const DevOracle& o, cg::cluster_group& cluster, int (*s_cnt)[BS_CLUSTER], int& phase,
                                                u32 j, i64 a, i64 b, double c, u32 k) {
  const unsigned crank = cluster.block_rank();
  if (a > b) return a;
  while (true) {
    const i64 S = b - a + 1;
    const i64 stride = (S + BS_WIDTH - 1) / BS_WIDTH;
    const i64 x = a + (i64)(crank * BS_THREADS + threadIdx.x) * stride;
    bool bad = false;  // a candidate inside the window whose cost still exceeds c
    if (x <= b) bad = !cost_leq(dev_cost<T>(o, j, (u32)x, k), c);
    const int mine = __syncthreads_count(bad);
    if (threadIdx.x < BS_CLUSTER) *cluster.map_shared_rank(&s_cnt[phase][crank], threadIdx.x) = mine;
    cluster.sync();
    int cf = 0;
#pragma unroll
    for (int p = 0; p < BS_CLUSTER; ++p) cf += s_cnt[phase][p];
    phase ^= 1;
    if (cf == 0) return a;                 // the first candidate already fits
    const i64 xf = a + (i64)(cf - 1) * stride;  // last candidate that does not fit
    if (stride == 1) return xf + 1;        // (= b + 1 if none fits)
    a = xf + 1;
    b = min(b, xf + stride);
    if (a > b) return b + 1;
  }
}

struct FlipResult {
  int probes, rounds;
};

// mode 0: FlipBisectCost (windows spl_lo / spl_hi, answer spl_lo); mode 1: LazyFlipBisectCost (no windows, answer spl_hi)
template <class T>
__device__ __forceinline__ void flip_bisect_body(const DevOracle& o, int (*s_cnt)[BS_CLUSTER], int K, double eps1, double c_lo, double c_hi, int lazy,
                                                 int* __restrict__ spl, int* __restrict__ spl_lo, int* __restrict__ spl_hi, int* __restrict__ probes_out) {
  cg::cluster_group cluster = cg::this_cluster();
  const bool cta0 = cluster.block_rank() == 0;
  const bool writer = cta0 && threadIdx.x == 0;
  const i64 n1 = (i64)o.n + 1;
  if (cta0)
    for (int t = 1 + threadIdx.x; t <= K + 1; t += blockDim.x) {
      spl_lo[t] = (t == K + 1) ? (int)n1 : 1;
      spl_hi[t] = (t == 1) ? 1 : (int)n1;
      spl[t] = (t == 1) ? 1 : (t == K + 1 ? (int)n1 : 0);
    }
  __threadfence();
  cluster.sync();
  int phase = 0, probes = 0;
  while (c_lo * eps1 < c_hi) {
    const double c = (c_lo + c_hi) / 2;
    ++probes;
    bool feas;
    if (!lazy) {  // BisectCost...:101-117
      bool chk = true;
      i64 j = 1;
      for (int k = 1; k <= K - 1; ++k) {
        const i64 a = max(j, (i64)__ldcg(spl_lo + k + 1));
        const i64 b = __ldcg(spl_hi + k + 1);
        const i64 r = wide_search_flip<T>(o, cluster, s_cnt, phase, (u32)j, a, b, c, (u32)k);
        if (writer) spl[k + 1] = (int)r;
        if (r > n1) {
          chk = false;
          if (cta0)
            for (int t = k + 1 + threadIdx.x; t <= K; t += blockDim.x) spl[t] = (int)n1;
          break;
        }
        j = r;
      }
      feas = chk && cost_leq(dev_cost<T>(o, (u32)j, (u32)n1, (u32)K), c);
    } else {  // LazyBisect...:96-124: every part ends at the first position (not before the previous end) where it fits
      feas = false;
      i64 j = 1;
      for (int k = 1; k <= K; ++k) {
        const i64 r = wide_search_flip<T>(o, cluster, s_cnt, phase, (u32)j, j, n1, c, (u32)k);
        if (r > n1) break;
        if (k == K) { feas = true; break; }
        if (writer) spl[k + 1] = (int)r;
        j = r;
      }
    }
    __syncthreads();
    if (feas) c_hi = c; else c_lo = c;
    if (cta0) {
      int* dst = nullptr;
      if (!lazy) dst = feas ? spl_lo : spl_hi;
      else if (feas) dst = spl_hi;
      if (dst) {
        for (int t = 1 + threadIdx.x; t <= K + 1; t += blockDim.x) dst[t] = (t == K + 1) ? (int)n1 : spl[t];
        __threadfence();
      }
    }
    cluster.sync();
  }
  if (writer) *probes_out = probes;
  cluster.sync();
}

// FlipBisectIndexBottleneckSplitter (BisectIndex...:87-166)
template <class T>
__device__ __forceinline__ void flip_bisect_index_body(const DevOracle& o, int (*s_cnt)[BS_CLUSTER], int K, double c_lo, double c_hi, int* __restrict__ spl,
                                                       int* __restrict__ spl_lo, int* __restrict__ spl_hi, int* __restrict__ probes_out) {
  cg::cluster_group cluster = cg::this_cluster();
  const bool cta0 = cluster.block_rank() == 0;
  const bool writer = cta0 && threadIdx.x == 0;
  const i64 n1 = (i64)o.n + 1;
  if (cta0)
    for (int t = 1 + threadIdx.x; t <= K + 1; t += blockDim.x) {
      spl_lo[t] = (t == K + 1) ? (int)n1 : 1;
      spl_hi[t] = (t == 1) ? 1 : (int)n1;
      spl[t] = (t == 1) ? 1 : (t == K + 1 ? (int)n1 : 0);
    }
  __threadfence();
  cluster.sync();
  int phase = 0, probes = 0;
  i64 sk = 1;
  for (int k = 1; k <= K; ++k) {
    i64 jp_hi = __ldcg(spl_hi + k + 1);
    i64 jp_lo = max(sk, (i64)__ldcg(spl_lo + k + 1));
    while (jp_lo <= jp_hi) {
      const i64 jp = (jp_lo + jp_hi) >> 1;
      const T c = dev_cost<T>(o, (u32)sk, (u32)jp, (u32)k);
      const double cd = (double)c;
      if (c_lo <= cd && cd < c_hi) {
        ++probes;
        bool chk = true;
        if (writer) spl[k + 1] = (int)jp;
        i64 j = jp;
        for (int kk = k + 1; kk <= K - 1; ++kk) {
          const i64 a = max(j, (i64)__ldcg(spl_lo + kk + 1));
          const i64 b = __ldcg(spl_hi + kk + 1);
          const i64 r = wide_search_flip<T>(o, cluster, s_cnt, phase, (u32)j, a, b, cd, (u32)kk);
          if (writer) spl[kk + 1] = (int)r;
          if (r > n1) {
            chk = false;
            if (cta0)
              for (int t = kk + 1 + threadIdx.x; t <= K; t += blockDim.x) spl[t] = (int)n1;
            break;
          }
          j = r;
        }
        const i64 ls = (k == K) ? sk : j, le = (k == K) ? jp : n1;
        const bool feas = chk && cost_leq(dev_cost<T>(o, (u32)ls, (u32)le, (u32)K), cd);
        __syncthreads();
        if (feas) { c_hi = cd; jp_lo = jp + 1; } else { c_lo = cd; jp_hi = jp - 1; }
        if (cta0) {
          int* dst = feas ? spl_lo : spl_hi;
          for (int t = 1 + threadIdx.x; t <= K + 1; t += blockDim.x) dst[t] = spl[t];
          __threadfence();
        }
        cluster.sync();
      } else if (cd >= c_hi) {
        jp_lo = jp + 1;
      } else {
        jp_hi = jp - 1;
      }
    }
    if (jp_lo > n1) break;
    if (writer) spl[k + 1] = (int)jp_lo;
    sk = jp_lo;
  }
  if (writer) *probes_out = probes;
  cluster.sync();
}

// ------------------------------------------------------------------------------------------------
// Batched solves (kernel "stripe_batch"): B independent problems of the four splitters above in one launch, one 8-CTA
// cluster per problem.  A solve is a latency chain of K part searches that occupies one cluster; a batch lets a K sweep,
// many matrices or the secondary models of a 2-D alternation fill the GPU instead of queueing one cluster at a time.
// ------------------------------------------------------------------------------------------------
struct StripeJob {
  int oracle;         // index into the batch's DevOracle table (one entry per distinct oracle)
  int method;         // CPB_SPLIT_BISECT_INDEX, CPB_SPLIT_FLIP_BISECT_COST, CPB_SPLIT_LAZY_FLIP_BISECT_COST or CPB_SPLIT_FLIP_BISECT_INDEX
  int K;
  int lazy;           // LazyFlipBisectCost
  double c_lo, c_hi;  // oracle_bound
  double eps1;        // 1 + eps (the FlipBisectCost forms)
  i64 spl, spl_lo, spl_hi, probes;  // offsets into the batch's int workspace
};

template <class T>
__global__ void __cluster_dims__(BS_CLUSTER, 1, 1) __launch_bounds__(BS_THREADS)
    k_stripe_batch(const DevOracle* __restrict__ oracles, const StripeJob* __restrict__ jobs, int* __restrict__ ws) {
  __shared__ int s_cnt[2][BS_CLUSTER];
  __shared__ DevOracle s_o;  // every cost evaluation reads the oracle's fields: keep them next to the SM, not in global memory
  static_assert(sizeof(DevOracle) % sizeof(u64) == 0, "DevOracle is copied in 8-byte words");
  const StripeJob jb = jobs[blockIdx.x / BS_CLUSTER];
  const u64* src = reinterpret_cast<const u64*>(oracles + jb.oracle);
  for (int t = threadIdx.x; t < (int)(sizeof(DevOracle) / sizeof(u64)); t += blockDim.x) reinterpret_cast<u64*>(&s_o)[t] = src[t];
  __syncthreads();
  int *spl = ws + jb.spl, *lo = ws + jb.spl_lo, *hi = ws + jb.spl_hi, *probes = ws + jb.probes;
  if (jb.method == CPB_SPLIT_BISECT_INDEX) bisect_index_body<T>(s_o, s_cnt, jb.K, jb.c_lo, jb.c_hi, spl, lo, hi, probes);
  else if (jb.method == CPB_SPLIT_FLIP_BISECT_INDEX) flip_bisect_index_body<T>(s_o, s_cnt, jb.K, jb.c_lo, jb.c_hi, spl, lo, hi, probes);
  else flip_bisect_body<T>(s_o, s_cnt, jb.K, jb.eps1, jb.c_lo, jb.c_hi, jb.lazy, spl, lo, hi, probes);
}

// ------------------------------------------------------------------------------------------------
// Streaming probe (kernel "probe_stream"): the device form of the reference's lazy probes
// (LazyBisectCostBottleneckSplitter.jl:194-229 connectivity, :323-359 monotonized symmetric).
// (Here the link array holds 1 + the CSC POSITION of the previous nonzero of the same row, so "previous column < j"
// is `prev <= first position of the part`; written `prev < j` below.)
// The reference streams cch[] = previous column of every nonzero and counts `cch[q] < j` for the
// current part start j; a part ends where the running cost first exceeds c.  Here one 8-CTA cluster
// per threshold streams the same link array in super-steps of register tiles: every lane stores its
// `prev < j` flags as one byte per group, a block scan gives each CTA's running count, and two st.async
// exchanges between the cluster's CTAs, completing on mbarriers, give the count at every column
// boundary inside the tile and the feasible boundaries of the whole cluster; all boundaries of the tile
// are tested at once.  No dominance index is needed for bisection at all.
// ------------------------------------------------------------------------------------------------
static constexpr int SP_THREADS = 1024;
#ifndef CPB_SP_VEC
#define CPB_SP_VEC 8
#endif
static constexpr int SP_VEC = CPB_SP_VEC;               // 128-bit loads per thread per register tile
static constexpr int SP_SUB = 2;                       // register tiles per super-step at most
static constexpr int SP_NVMAX = SP_VEC * SP_SUB;       // 128-bit loads per thread per super-step at most
static constexpr int SP_CE = SP_THREADS * SP_VEC * 4;  // 32768 elements per CTA per register tile
static constexpr int SP_GROUPS = SP_NVMAX * 32;        // 128-element groups per CTA (one warp-wide uint4 load each) at most

// `prev < j` count among the first x elements of this CTA's slice, from the per-group flags stored as one byte per lane (bit k
// of byte l = element 4 l + k of the group; 8 words per group): every thread stores the nibble of its own four compares, no
// warp vote (VOTE runs on the SM's one address-divergence unit: 1024 votes per super-step were the tile phase's limiter).
__device__ __forceinline__ u32 stream_prefix_nib(const u32* s_mask, const u32* s_cum, u32 x) {
  const u32 g = x >> 7, r = x & 127u;
  u32 cnt = s_cum[g];
  const uint4 a = *reinterpret_cast<const uint4*>(&s_mask[g * 8]);
  const uint4 b = *reinterpret_cast<const uint4*>(&s_mask[g * 8 + 4]);
  const u32 w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  const u32 full = r >> 4, q8 = ((r & 15u) >> 2) * 8u, t = r & 3u;
  const u32 msk = ((1u << q8) - 1u) | (((1u << t) - 1u) << q8);
#pragma unroll
  for (u32 i = 0; i < 8; ++i) cnt += __popc(i < full ? w[i] : (i == full ? (w[i] & msk) : 0u));
  return cnt;
}

struct DevStream {
  const u32* prev;    // [Ne] 1 + position of the previous nonzero of the same row (0 = none): "its column lies left of the part"
                      //      is simply prev <= first position of the part
  const u32* colq;    // [ceil(Ne / LS_COLQ) + 1] 0-based column of every LS_COLQ-th element (LinkStream::colq)
  const u32* P;       // element offsets of the column boundaries, 1 <= x <= n+1
  const u32* Wt;      // prefix of the pin-like term, 1 <= x <= n+1
  u32 Ne, n;
  int same_w;         // Wt == P
  double cf[4];
  i64 ci[4];
};

template <class T> struct StreamCoef;
template <> struct StreamCoef<i64> { static __device__ __forceinline__ i64 get(const DevStream& s, int t) { return s.ci[t]; } };
template <> struct StreamCoef<double> { static __device__ __forceinline__ double get(const DevStream& s, int t) { return s.cf[t]; } };
template <class T> __device__ __forceinline__ T stream_cost(const DevStream& s, i64 nv, i64 w, i64 g) {
  using C = StreamCoef<T>;  // alpha + n_vertices * b_vertex + n_pins * b_pin + n_nets * b_net, left to right
  return C::get(s, 0) + (T)nv * C::get(s, 1) + (T)w * C::get(s, 2) + (T)g * C::get(s, 3);
}

// ---- cluster exchange primitives (PTX) ----
__device__ __forceinline__ u32 smem_addr(const void* p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ u32 map_peer(u32 addr, u32 rank) {
  u32 r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_init(u32 bar, u32 count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(u32 bar, u32 bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// A wait that never completes -- a protocol bug -- traps after ~2 s instead of hanging the GPU, after leaving a record
// (which wait, where) in a host-mapped buffer that bisect_advance appends to the error message.
__device__ unsigned long long* g_probe_dbg = nullptr;
__device__ __noinline__ void probe_wait_failed(u32 tag, u32 a, u32 b, u32 c, u32 d) {
  unsigned long long* g = g_probe_dbg;
  if (g) {
    unsigned cr;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(cr));
    // the first record wins; every field travels in one 64-bit system-scope atomic (plain stores may not leave the SM
    // before the trap): word 0 = 1 | tag << 4 | crank << 8 | block << 12 | tid << 28, words 1..2 = (a, b), (c, d)
    const unsigned long long w0 = 1ull | ((unsigned long long)(tag & 15u) << 4) | ((unsigned long long)(cr & 15u) << 8) |
                                  ((unsigned long long)(blockIdx.x & 0xffffu) << 12) | ((unsigned long long)(threadIdx.x & 0xfffu) << 28);
    if (atomicCAS_system(g, 0ull, w0) == 0ull) {
      atomicExch_system(g + 1, ((unsigned long long)a << 32) | b);
      atomicExch_system(g + 2, ((unsigned long long)c << 32) | d);
      __threadfence_system();
    }
    // give the record time to reach the host before the context dies
    const long long t0 = clock64();
    while (clock64() - t0 < 2000000) {}
  }
  __trap();
}
__device__ __forceinline__ void mbar_wait_cluster(u32 bar, u32 parity, u32 tag = 0, u32 a = 0, u32 b = 0, u32 c = 0, u32 d = 0) {  // peers' st.async
  u32 ok = 0;
  long long t0 = 0;
  while (true) {
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) break;
    const long long t = clock64();
    if (t0 == 0) t0 = t;
    else if (t - t0 > 4000000000ll) probe_wait_failed(tag, a, b, c, d);
  }
}
__device__ __forceinline__ void st_async_u32(u32 remote_addr, u32 v, u32 remote_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.u32 [%0], %1, [%2];" ::"r"(remote_addr), "r"(v), "r"(remote_bar) : "memory");
}
__device__ __forceinline__ void st_async_v4(u32 remote_addr, u32 a, u32 b, u32 c, u32 d, u32 remote_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(remote_addr), "r"(a), "r"(b),
               "r"(c), "r"(d), "r"(remote_bar) : "memory");
}

#ifdef CPB_PROBE_TIMING
__device__ unsigned long long g_probe_t[16];
__device__ unsigned long long g_probe_n;
__device__ unsigned long long g_probe_parts[4];  // per slot 0..3: parts started
__device__ unsigned long long g_probe_node[16][4];  // per slot: cycles of its cluster, super-steps, parts, launches
// (accumulated in shared memory by one thread and flushed at the end: a global read-modify-write per mark costs an L2 round trip)
#define PT(i) do { if (node == node_base && crank == 0 && tid == 0) { unsigned long long _t = clock64(); s_pt[i] += _t - t_last; t_last = _t; } } while (0)
#else
#define PT(i) do {} while (0)
#endif

// 0-based columns of the elements e1, e2 < Ne (use1 / use2: which are wanted): the largest c with P[c + 1] <= e, searched by the
// whole warp (32 probes per step, counted with a warp reduction -- no vote) between the columns the per-128-element table
// brackets it with; both searches advance together so that their loads overlap.  Warp-uniform arguments.
__device__ __forceinline__ void stream_cols_of(const DevStream& s, bool use1, u32 e1, bool use2, u32 e2, int lane, u32& c1, u32& c2) {
  u32 lo1 = 0, hi1 = 0, lo2 = 0, hi2 = 0;
  if (use1) { lo1 = __ldg(s.colq + e1 / LS_COLQ); hi1 = __ldg(s.colq + e1 / LS_COLQ + 1); }  // (behind the end the table holds n - 1)
  if (use2) { lo2 = __ldg(s.colq + e2 / LS_COLQ); hi2 = __ldg(s.colq + e2 / LS_COLQ + 1); }
  while (hi1 > lo1 || hi2 > lo2) {
    const u32 st1 = (hi1 - lo1 + 31u) / 32u, st2 = (hi2 - lo2 + 31u) / 32u;
    const u64 p1 = (u64)lo1 + (u64)(lane + 1) * st1, p2 = (u64)lo2 + (u64)(lane + 1) * st2;  // this lane's probes; those that hold form a prefix
    const bool ok1 = hi1 > lo1 && p1 <= hi1 && __ldg(s.P + p1 + 1) <= e1;
    const bool ok2 = hi2 > lo2 && p2 <= hi2 && __ldg(s.P + p2 + 1) <= e2;
    const u32 cnt = __reduce_add_sync(0xffffffffu, (ok1 ? 1u : 0u) | (ok2 ? 0x10000u : 0u));
    if (hi1 > lo1) { const u32 nlo = lo1 + (cnt & 0xffffu) * st1; hi1 = (u32)min((u64)hi1, (u64)nlo + st1 - 1); lo1 = nlo; }
    if (hi2 > lo2) { const u32 nlo = lo2 + (cnt >> 16) * st2; hi2 = (u32)min((u64)hi2, (u64)nlo + st2 - 1); lo2 = nlo; }
  }
  c1 = lo1;
  c2 = lo2;
}

// The two exchanges of a super-step are remote st.async stores that complete a transaction count on every peer's mbarrier
// (no barrier.cluster, no fence in front of it, no L1 invalidation).
template <class T>
__global__ void __cluster_dims__(BS_CLUSTER, 1, 1) __launch_bounds__(SP_THREADS, 1)
    k_probe_stream(const __grid_constant__ DevStream s, int K, double eps1, const BisectState* __restrict__ st,
                   int* __restrict__ node_spl, int* __restrict__ node_res, double* __restrict__ node_c,
                   const int* __restrict__ node_ids, int node_base) {
  __shared__ __align__(16) u32 s_mask[SP_GROUPS * 8 + 8];  // one byte per lane and group: the lane's four `prev <= e0` flags
  __shared__ u32 s_cum[SP_GROUPS + 1];
  __shared__ double s_c;
  __shared__ int s_valid;
  __shared__ u32 s_xa[2][BS_CLUSTER];  // per-CTA `prev < j` totals of the tile
  __shared__ __align__(16) u32 s_xv[2][BS_CLUSTER][4];  // per CTA (feasible boundaries, boundaries, P and Wt at the last feasible one)
  __shared__ __align__(8) unsigned long long s_mb[2][2];  // [exchange][super-step parity]
  __shared__ u32 s_pj[2 * SP_THREADS];    // (P, Wt) of every thread's boundary candidate, pass 1 | pass 2
  __shared__ u32 s_w[2 * SP_THREADS];
  __shared__ u32 s_wtot[32];              // per-warp `prev < j` totals of the tile
  __shared__ u32 s_red[2][4];             // single-pass boundary test: (feasible boundaries, max P, max Wt) of the CTA
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned crank = cluster.block_rank();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int node = node_base + blockIdx.x / BS_CLUSTER;
  const bool writer = crank == 0 && tid == 0;
  if (tid == 0) {
    s_valid = node_threshold(st, eps1, node_ids[node], &s_c);
    for (int k = 0; k < 8; ++k) s_mask[SP_GROUPS * 8 + k] = 0;
    for (int k = 0; k < 4; ++k) { s_red[0][k] = 0; s_red[1][k] = 0; }
    for (int x = 0; x < 2; ++x)
      for (int p = 0; p < 2; ++p) mbar_init(smem_addr(&s_mb[x][p]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (!s_valid) {
    if (writer) node_res[node] = 0;
    return;
  }
  cluster.sync();  // every CTA's mbarriers exist before a peer's st.async can reach them
  u32 sstep = 0;
#ifdef CPB_PROBE_TIMING
  __shared__ unsigned long long s_pt[16];
  if (tid == 0) for (int i = 0; i < 16; ++i) s_pt[i] = 0;
  const long long t_node0 = clock64();
  unsigned long long t_last = clock64();
  u32 parts_run = 0;
#endif
  const double c = s_c;
  const u32 n1 = s.n + 1;
  const u32 Ne = s.Ne;
  u32 nv = SP_VEC, nv_est = SP_VEC;  // 128-bit loads per thread in the next super-step: adapted to the previous parts' sizes
  int* spl = node_spl + (size_t)node * (K + 2);
  if (writer) { spl[1] = 1; spl[K + 1] = (int)n1; }
  int ph = 0;
  u32 j = 1;
  bool broke = false, feasible = false;
  u32 pcur = __ldg(s.P + 1), wcur = __ldg(s.Wt + 1);  // P[j], Wt[j] of the current part start, carried from the boundary tests
  for (int k = 1; k <= K; ++k) {
    // largest boundary r >= j with c(j, r) <= c
    if (!cost_leq(stream_cost<T>(s, 0, 0, 0), c)) { broke = true; break; }  // even the empty part exceeds c
    const u32 e0 = pcur;
    const i64 wj = (i64)wcur;
#ifdef CPB_PROBE_TIMING
    parts_run += 1;
#endif
    u32 jlast = j;
    u32 grun = 0;
    bool first = true, missed = false;
    PT(10);
    for (u32 e_tile = e0 & ~3u;;) {  // 16-byte aligned tiles; elements left of e0 are masked out
      const u32 CE = (u32)SP_THREADS * 4u * nv;  // elements of this CTA in this super-step
      const u32 TE = CE * BS_CLUSTER;
      const u32 ngroups = nv * 32u;
#ifdef CPB_PROBE_TIMING
      PT(6);  // between the super-steps (part bookkeeping)
#endif
      const u32 e_c = e_tile + crank * CE;
      // ---- column boundaries whose element offset falls into (e_c, e_c + CE] ----
      u32 ja = 0, jb = 0;  // (found below, while the tile's loads are in flight)
      // ---- flags of `prev <= e0`: each warp owns nv consecutive 128-element groups (one warp-wide 128-bit load per group);
      //      every lane stores the nibble of its four compares as one byte, the group totals come from two packed warp
      //      reductions.  (Round 1 formed the masks with 4 ballots per group: 1024 VOTEs per CTA and super-step on the SM's one
      //      address-divergence unit -- ~3 cycles each, measured with tools/ubench -- were what bounded this phase.) ----
      u32 wsum = 0;
      // A part longer than one register tile (8 vector loads per thread) takes up to SP_SUB tiles in the same super-step:
      // the flags live in shared memory, only the loads repeat -- one more load phase instead of a whole second super-step
      // with its two exchanges (parts of 262 k - 524 k elements: config 5, a quarter of config 3's parts).
      unsigned char* const s_nib = reinterpret_cast<unsigned char*>(s_mask);
      u32 pk[SP_SUB * 2];  // flag counts of the warp's groups, one byte per group (<= 128 each)
#pragma unroll
      for (int i = 0; i < SP_SUB * 2; ++i) pk[i] = 0;
#pragma unroll
      for (int sub = 0; sub < SP_SUB; ++sub) {
        if ((u32)sub * SP_VEC >= nv) break;
        // all loads of the tile are issued before the first compare (one exposed memory latency instead of nv)
        uint4 pv[SP_VEC];
#pragma unroll
        for (int v = 0; v < SP_VEC; ++v) {
          pv[v] = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);  // (beyond the end: never counted)
          if ((u32)(sub * SP_VEC + v) < nv) {
            const u32 idx = e_c + (warp * nv + sub * SP_VEC + v) * 128 + lane * 4;
            if ((u64)idx + 4 <= Ne) {
              pv[v] = __ldg(reinterpret_cast<const uint4*>(s.prev + idx));
            } else {
              if (idx < Ne) pv[v].x = __ldg(s.prev + idx);
              if (idx + 1 < Ne) pv[v].y = __ldg(s.prev + idx + 1);
              if (idx + 2 < Ne) pv[v].z = __ldg(s.prev + idx + 2);
            }
          }
        }
        if (sub == 0) {  // the columns of the slice's two ends: two short cooperative searches behind the tile's loads
          const bool head = first && crank == 0;
          const bool want_a = !head && e_c < Ne, want_b = (head || e_c < Ne) && (u64)e_c + CE < Ne;
          u32 ca = 0, cb = 0;
          stream_cols_of(s, want_a, e_c, want_b, e_c + CE, lane, ca, cb);
          ja = head ? j + 1 : (e_c < Ne ? ca + 2 : n1 + 1);
          jb = (e_c >= Ne && !head) ? 0u : (((u64)e_c + CE >= Ne) ? n1 : cb + 1);
        }
#pragma unroll
        for (int v = 0; v < SP_VEC; ++v) {
          if ((u32)(sub * SP_VEC + v) >= nv) break;
          const u32 g = warp * nv + sub * SP_VEC + v;
          const u32 gbase = e_c + g * 128;  // first element of the group (warp-uniform)
          u32 nib;
          if (gbase >= e0) {
            nib = (u32)(pv[v].x <= e0) | ((u32)(pv[v].y <= e0) << 1) | ((u32)(pv[v].z <= e0) << 2) | ((u32)(pv[v].w <= e0) << 3);
          } else {  // the group holding the part's first element: mask what lies in front of it
            const u32 idx = gbase + lane * 4;
            nib = (u32)(pv[v].x <= e0 && idx + 0 >= e0) | ((u32)(pv[v].y <= e0 && idx + 1 >= e0) << 1) | ((u32)(pv[v].z <= e0 && idx + 2 >= e0) << 2) |
                  ((u32)(pv[v].w <= e0 && idx + 3 >= e0) << 3);
          }
          s_nib[g * 32 + lane] = (unsigned char)nib;
          pk[(sub * SP_VEC + v) >> 2] += (u32)__popc(nib) << (8 * (v & 3));
        }
      }
      {
        // lane v: flags in the warp's groups before group v (prefix inside the warp's run; the warp's base is added after the barrier)
        u32 pre = 0;
#pragma unroll
        for (int i = 0; i < SP_SUB * 2; ++i) {
          if ((u32)(4 * i) >= nv) break;
          const u32 R = __reduce_add_sync(0xffffffffu, pk[i]);
          const u32 m = lane >= 4 * (i + 1) ? 0xffffffffu : (lane <= 4 * i ? 0u : ((1u << (8 * (lane - 4 * i))) - 1u));
          pre = __dp4a(R & m, 0x01010101u, pre);
          wsum = __dp4a(R, 0x01010101u, wsum);
        }
        if (lane < (int)nv) s_cum[warp * nv + lane] = pre;
      }
      if (lane == 0) s_wtot[warp] = wsum;
      PT(0);
      __syncthreads();
      PT(1);
      // ---- every warp adds the totals of the warps before it to its own groups' prefixes; warp 0 also forms the CTA
      //      total.  The __syncthreads below orders these writes for the boundary phase. ----
      u32 tot_c = 0;
      {
        const u32 t = s_wtot[lane];
        const u32 wbase = __reduce_add_sync(0xffffffffu, lane < warp ? t : 0u);
        if (lane < (int)nv) s_cum[warp * nv + lane] += wbase;
        if (warp == 0) {
          tot_c = __reduce_add_sync(0xffffffffu, t);
          if (lane == 0) {
            s_cum[ngroups] = tot_c;
            // sentinel masks behind the last group (prefix lookups at x == CE)
            *reinterpret_cast<uint4*>(&s_mask[ngroups * 8]) = make_uint4(0u, 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(&s_mask[ngroups * 8 + 4]) = make_uint4(0u, 0u, 0u, 0u);
          }
        }
      }
      PT(2);
      const u32 xpar = (sstep >> 1) & 1u;
      if (tid == 0) { mbar_expect_tx(smem_addr(&s_mb[0][ph]), 4u * BS_CLUSTER); mbar_expect_tx(smem_addr(&s_mb[1][ph]), 16u * BS_CLUSTER); }
      if (tid < BS_CLUSTER) st_async_u32(map_peer(smem_addr(&s_xa[ph][crank]), tid), tot_c, map_peer(smem_addr(&s_mb[0][ph]), tid));
      const u32 nb = (jb >= ja) ? jb - ja + 1 : 0;
      // thread t owns the (at most 4) consecutive boundaries [t * per, (t + 1) * per) when the CTA has at most 4096 of
      // them: all loaded up front (one memory latency), before the barrier completes
      const bool few = nb > 0 && nb <= 4u * SP_THREADS;
      const u32 per = (nb + SP_THREADS - 1) / SP_THREADS;
      const u32 b0 = (u32)tid * per;
      const u32 mine = (few && b0 < nb) ? min(per, nb - b0) : 0u;
      u32 pjv[4], wv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (i < (int)mine) {
          pjv[i] = __ldg(s.P + ja + b0 + i);
          wv[i] = s.same_w ? pjv[i] : __ldg(s.Wt + ja + b0 + i);
        }
      __syncthreads();  // s_cum (every warp added its base) is complete for the boundary phase
      mbar_wait_cluster(smem_addr(&s_mb[0][ph]), xpar, 5u, sstep, nv, e0, e_tile);
      PT(3);
      u32 base_c = 0, tile_tot = 0;
#pragma unroll
      for (int p = 0; p < BS_CLUSTER; ++p) {
        const u32 v = s_xa[ph][p];
        if (p < (int)crank) base_c += v;
        tile_tot += v;
      }
      auto feasible_pw = [&](u32 jp, u32 pj, u32 w) -> bool {
        const u32 g = grun + base_c + stream_prefix_nib(s_mask, s_cum, pj - e_c);
        return cost_leq(stream_cost<T>(s, (i64)jp - (i64)j, (i64)w - wj, (i64)g), c);
      };
      // monotone costs: the feasible boundaries of this CTA form a prefix [ja, ja + cnt); every thread stashes the
      // (P, Wt) of its candidate so the next part can start without reloading them.
      u32 cnt = 0, lastp = 0, lastw = 0;
      if (tid == 0) { s_red[ph ^ 1][0] = 0; s_red[ph ^ 1][1] = 0; s_red[ph ^ 1][2] = 0; }  // the next super-step's accumulators
      if (few) {
        // every thread tests its LAST boundary; the first thread whose last boundary fails holds the crossing and tests
        // its remaining ones from registers.
        bool ok = false;
        if (mine > 0) {
          u32 pl = pjv[0], wl = wv[0];
#pragma unroll
          for (int i = 1; i < 4; ++i)
            if (i < (int)mine) { pl = pjv[i]; wl = wv[i]; }
          s_pj[tid] = pl;
          s_w[tid] = wl;
          ok = feasible_pw(ja + b0 + mine - 1, pl, wl);
        }
        const int ct = __syncthreads_count(ok);  // threads 0 .. ct-1 are feasible throughout
        cnt = min((u32)ct * per, nb);
        if (ct > 0) { lastp = s_pj[ct - 1]; lastw = s_w[ct - 1]; }
        if (per > 1) {
          if (tid == ct && mine > 1) {
            u32 c2 = 0, lp = 0, lw = 0;
#pragma unroll
            for (int i = 0; i < 3; ++i)
              if (i < (int)mine - 1 && c2 == (u32)i && feasible_pw(ja + b0 + i, pjv[i], wv[i])) { c2 = i + 1; lp = pjv[i]; lw = wv[i]; }
            s_red[ph][0] = c2;
            s_red[ph][1] = lp;
            s_red[ph][2] = lw;
          }
          __syncthreads();
          const u32 c2 = s_red[ph][0];
          if (c2 > 0) { cnt += c2; lastp = s_red[ph][1]; lastw = s_red[ph][2]; }
        }
      } else if (nb > 0) {
        const u32 stride = (nb + SP_THREADS - 1) / SP_THREADS;
        const u32 t0 = (u32)tid * stride;
        bool ok = false;
        if (t0 < nb) {
          const u32 pj = __ldg(s.P + ja + t0);
          const u32 w = s.same_w ? pj : __ldg(s.Wt + ja + t0);
          s_pj[tid] = pj;
          s_w[tid] = w;
          ok = feasible_pw(ja + t0, pj, w);
        }
        const int ct = __syncthreads_count(ok);
        if (ct > 0) {
          const u32 base = (u32)(ct - 1) * stride;  // last feasible probe
          cnt = base + 1;
          lastp = s_pj[ct - 1];
          lastw = s_w[ct - 1];
          if (stride > 1) {
            const u32 off = base + 1 + tid;
            ok = false;
            if (tid < stride - 1 && off < nb) {
              const u32 pj = __ldg(s.P + ja + off);
              const u32 w = s.same_w ? pj : __ldg(s.Wt + ja + off);
              s_pj[SP_THREADS + tid] = pj;
              s_w[SP_THREADS + tid] = w;
              ok = feasible_pw(ja + off, pj, w);
            }
            const int c2 = __syncthreads_count(ok);
            if (c2 > 0) {
              cnt += c2;
              lastp = s_pj[SP_THREADS + c2 - 1];
              lastw = s_w[SP_THREADS + c2 - 1];
            }
          }
        }
      }
      PT(4);
      u32 feas = 0, nbs = 0;
      if (tid < BS_CLUSTER) st_async_v4(map_peer(smem_addr(&s_xv[ph][crank][0]), tid), cnt, nb, lastp, lastw, map_peer(smem_addr(&s_mb[1][ph]), tid));
      mbar_wait_cluster(smem_addr(&s_mb[1][ph]), xpar, 6u, sstep, nv, e0, e_tile);
      PT(5);
#pragma unroll
      for (int p = 0; p < BS_CLUSTER; ++p) {
        const uint4 q = *reinterpret_cast<const uint4*>(&s_xv[ph][p][0]);
        feas += q.x;
        nbs += q.y;
        if (q.x > 0) { pcur = q.z; wcur = q.w; }  // the last CTA with a feasible boundary wins
      }
      PT(7);
      ++sstep;
      ph ^= 1;
      first = false;
      jlast += feas;
      if (feas < nbs) break;                   // the cost crossed c inside this tile
      if ((u64)e_tile + TE >= Ne) break;       // streamed to the end: jlast == n + 1
      grun += tile_tot;
      e_tile += TE;
      nv = SP_NVMAX;                           // the part is longer than estimated: full-size tiles from here on
      missed = true;
    }
    {  // size the next part's first tile from this part (+1/8 slack); a miss (second super-step needed) resets
       // the estimate to the full tile, from where it shrinks by one vector load per part at most
      const u32 elems = pcur - e0;
      const u32 want = (elems + (elems >> 3) + 3u) / ((u32)SP_THREADS * 4u * BS_CLUSTER) + 1u;
      nv_est = missed ? (u32)SP_NVMAX : max(min(max(want, 2u), (u32)SP_NVMAX), nv_est > 2u ? nv_est - 1u : 2u);
      nv = nv_est;
    }
    PT(8);
    if (k == K) { feasible = (jlast == n1); break; }
    if (jlast == n1) {  // every column is placed: the remaining parts are empty (their cost was tested at the loop top)
      if (writer)
        for (int t = k + 1; t <= K; ++t) spl[t] = (int)n1;
      feasible = true;
      break;
    }
    if (writer) spl[k + 1] = (int)jlast;
    j = jlast;
    PT(9);
  }
  if (writer) {
    node_c[node] = c;
    node_res[node] = (!broke && feasible) ? 2 : 1;
#ifdef CPB_PROBE_TIMING
    if (node - node_base < 16) {
      unsigned long long* g = g_probe_node[node - node_base];
      g[0] += (unsigned long long)(clock64() - t_node0); g[1] += sstep; g[2] += parts_run; g[3] += 1;
    }
    if (node == node_base) {
      for (int i = 0; i < 16; ++i) g_probe_t[i] += s_pt[i];
      g_probe_n += sstep;
    }
#endif
  }
  cluster.sync();
}

__global__ void k_count_zero(const u32* __restrict__ v, size_t n, u32* __restrict__ out) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  u32 c = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) c += v[i] == 0u;
  c = __reduce_add_sync(0xffffffffu, c);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

// walks the probed subtree by feasibility (BisectCost...:53-59)
__global__ void k_bisect_advance(int K, int P, double eps1, BisectState* st, int* __restrict__ hint_lo, int* __restrict__ hint_hi,
                                 int* __restrict__ best, const int* __restrict__ node_spl, const int* __restrict__ node_res,
                                 const double* __restrict__ node_c, const int* __restrict__ node_ids) {
  if (st->done) return;
  int heap = 0;
  while (true) {
    int node = -1;  // slot holding tree node `heap`; the walk leaves the probed set -> the next round continues from here
    for (int t = 0; t < P; ++t)
      if (node_ids[t] == heap) { node = t; break; }
    if (node < 0) break;
    const int res = node_res[node];
    if (res == 0) {
      if (threadIdx.x == 0) st->done = 1;
      return;
    }
    const int* spl = node_spl + (size_t)node * (K + 2);
    if (res == 2) {
      for (int t = 1 + threadIdx.x; t <= K + 1; t += blockDim.x) { best[t] = spl[t]; hint_hi[t] = spl[t]; }
      if (threadIdx.x == 0) { st->c_hi = node_c[node]; st->probes += 1; }
      heap = 2 * heap + 1;
    } else {
      for (int t = 1 + threadIdx.x; t <= K + 1; t += blockDim.x) hint_lo[t] = spl[t];
      if (threadIdx.x == 0) { st->c_lo = node_c[node]; st->probes += 1; }
      heap = 2 * heap + 2;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    st->rounds += 1;
    if (!(st->c_lo * eps1 < st->c_hi)) st->done = 1;
  }
}

// pulls a read-only buffer into L2 ahead of the latency-bound probes (one prefetch per 128-byte line)
__global__ void k_l2_prefetch(const char* __restrict__ p, size_t bytes) {
  const size_t stride = (size_t)gridDim.x * blockDim.x * 128;
  for (size_t off = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 128; off < bytes; off += stride)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p + off));
}

__global__ void k_bisect_init(int K, int n1, int* hint_lo, int* hint_hi, int* best) {
  for (int t = 1 + threadIdx.x; t <= K + 1; t += blockDim.x) {
    hint_lo[t] = (t == K + 1) ? n1 : 1;
    hint_hi[t] = (t == 1) ? 1 : n1;
    best[t] = (t == 1) ? 1 : n1;
  }
}

static int env_int(const char* name, int dflt) {
  const char* s = std::getenv(name);
  return s ? std::atoi(s) : dflt;
}

// nets(1, n+1) = number of non-empty rows = links equal to 0 (ConnectivityCosts.jl:32 needs ocl(1, n+1))
i64 count_first_occurrences(const LinkStream& ls) {
  // counted while the links were written (k_lt_link, or the one-sweep link kernels of the k_link_prev phase)
  u32 h = 0;
  CPB_CUDA(cudaMemcpyAsync(&h, ls.first_count.get(), sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  return (i64)h;
}

// ---- a cheap upper bound on the optimal bottleneck, used ONLY to decide which thresholds of the bisection tree are
//      worth probing speculatively (plan_round below; the returned split vector never depends on it).  The columns are
//      cut where U(x) = b_vertex x + b_pin Wt[x] + b_net P[x] (the cost with every pin counted as a new net) crosses
//      k/K of its total; the bottleneck of that partition, evaluated exactly with one fused pass over the links, bounds
//      the optimum from above.
__device__ __forceinline__ double ub_weight(const DevStream& s, const double* cf, u32 x) {
  return cf[1] * (double)x + cf[2] * (double)__ldg(s.Wt + x) + cf[3] * (double)__ldg(s.P + x);
}
__global__ void k_ub_splits(const __grid_constant__ DevStream s, int is_float, int K, int* __restrict__ spl, u32* __restrict__ cnt) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;  // spl[k], k = 0..K (0-based parts, 1-based columns)
  if (k > K) return;
  double cf[4];
  for (int t = 0; t < 4; ++t) cf[t] = is_float ? s.cf[t] : (double)s.ci[t];
  if (!(cf[1] + cf[2] + cf[3] > 0)) { cf[1] = 1; cf[2] = 0; cf[3] = 0; }
  const u32 n1 = s.n + 1;
  const double u0 = ub_weight(s, cf, 1), u1 = ub_weight(s, cf, n1);
  const double target = u0 + (u1 - u0) * ((double)k / (double)K);
  u32 lo = 1, hi = n1;  // smallest x with U(x) >= target
  while (lo < hi) {
    const u32 mid = lo + ((hi - lo) >> 1);
    if (ub_weight(s, cf, mid) >= target) hi = mid; else lo = mid + 1;
  }
  spl[k] = (k == 0) ? 1 : (k == K ? (int)n1 : (int)lo);
  if (k < K) cnt[k] = 0;
}
__global__ void __launch_bounds__(256) k_ub_count(const __grid_constant__ DevStream s, const int* __restrict__ spl, u32* __restrict__ cnt,
                                                  const int* __restrict__ stop = nullptr) {
  if (stop && *stop) return;
  const int k = blockIdx.y;
  const u32 j = (u32)spl[k];
  const u32 e0 = __ldg(s.P + j), e1 = __ldg(s.P + (u32)spl[k + 1]);
  u32 c = 0;
  const u32 stride = gridDim.x * blockDim.x;
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  // 128-bit loads over the 16-byte aligned middle of [e0, e1), four in flight per thread; scalar head and tail
  const u32 a0 = min((e0 + 3u) & ~3u, e1), a1 = max(e1 & ~3u, a0);
  if (t < a0 - e0) c += __ldg(s.prev + e0 + t) <= e0;
  if (t < e1 - a1) c += __ldg(s.prev + a1 + t) <= e0;
  const uint4* v4 = reinterpret_cast<const uint4*>(s.prev + a0);
  const u32 nvec = (a1 - a0) >> 2;
  u32 i = t;
  for (; (u64)i + 3ull * stride < nvec; i += 4 * stride) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = __ldg(v4 + i + (u32)u * stride);
#pragma unroll
    for (int u = 0; u < 4; ++u) c += (v[u].x <= e0) + (v[u].y <= e0) + (v[u].z <= e0) + (v[u].w <= e0);
  }
  for (; i < nvec; i += stride) {
    const uint4 v = __ldg(v4 + i);
    c += (v.x <= e0) + (v.y <= e0) + (v.z <= e0) + (v.w <= e0);
  }
  c = __reduce_add_sync(0xffffffffu, c);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(&cnt[k], c);
}
__global__ void k_ub_zero(u32* __restrict__ cnt, int K, const int* __restrict__ stop) {
  if (*stop) return;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < K) cnt[k] = 0;
}
__global__ void k_ub_max(const __grid_constant__ DevStream s, int is_float, int K, const int* __restrict__ spl, const u32* __restrict__ cnt,
                         double* __restrict__ out) {
  __shared__ double sm[32];
  double cf[4];
  for (int t = 0; t < 4; ++t) cf[t] = is_float ? s.cf[t] : (double)s.ci[t];
  double best = 0;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const u32 a = (u32)spl[k], b = (u32)spl[k + 1];
    const double c = cf[0] + (double)(b - a) * cf[1] + ((double)__ldg(s.Wt + b) - (double)__ldg(s.Wt + a)) * cf[2] + (double)cnt[k] * cf[3];
    best = fmax(best, c);
  }
  for (int o = 16; o > 0; o >>= 1) best = fmax(best, __shfl_xor_sync(0xffffffffu, best, o));
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = best;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) best = fmax(best, sm[w]);
    out[0] = best;
  }
}

// ---- refinement of the bounding partition (round 2).  A partition whose parts all cost the same is optimal for a cost that
//      grows with the part (a partition with a smaller bottleneck would have to end every part earlier, including the last),
//      so the bound is tight when the exact part costs are balanced.  One refinement step rescales the additive weight U
//      inside every part so that the part weighs its exact cost, and cuts the rescaled weight greedily at the smallest
//      threshold that needs at most K parts (a column heavier than the mean share stays alone -- equal-share cuts cannot do
//      that); the new partition is evaluated exactly by k_ub_count again.  On R-MAT the first bound is 20-40 % above the
//      optimum, one or two steps bring it within ~1 % (tools/ub_refine_proto.py), which lets one round of speculated
//      thresholds finish the bisection.  Only the plan depends on the bound.
static constexpr int UB_G = 32768;      // grid points of the rescaled weight (uniform in weight)
static constexpr int UB_T = 1024;       // candidate thresholds of the parametric search, one per thread
static constexpr int UB_KMAX = 4096;    // parts (the candidates' cut lists live in a [UB_T][K + 1] scratch array)
struct UbCtl { double best; double total; double tlo; double tstar; int stop; int pad; };

// exact part costs -> ctl.best = min(ctl.best, bottleneck); prefix S[k] of (cost - alpha), per-part scale of U
__global__ void __launch_bounds__(1024) k_ub_prepare(const __grid_constant__ DevStream s, int is_float, int K, const int* __restrict__ spl,
                                                     const u32* __restrict__ cnt, double* __restrict__ S, double* __restrict__ scale,
                                                     UbCtl* __restrict__ ctl, double* __restrict__ out, int first, double tol) {
  __shared__ double sm[32];
  __shared__ double s_carry;
  double cf[4];
  for (int t = 0; t < 4; ++t) cf[t] = is_float ? s.cf[t] : (double)s.ci[t];
  double ucf[4] = {cf[0], cf[1], cf[2], cf[3]};
  if (!(ucf[1] + ucf[2] + ucf[3] > 0)) { ucf[1] = 1; ucf[2] = 0; ucf[3] = 0; }
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid == 0) s_carry = 0;
  double best = 0;
  int single = 0;  // the costliest part seen by this thread is one column wide
  __syncthreads();
  for (int k0 = 0; k0 < K; k0 += 1024) {
    const int k = k0 + tid;
    double wk = 0;
    if (k < K) {
      const u32 a = (u32)spl[k], b = (u32)spl[k + 1];
      const double c = cf[0] + (double)(b - a) * cf[1] + ((double)__ldg(s.Wt + b) - (double)__ldg(s.Wt + a)) * cf[2] + (double)cnt[k] * cf[3];
      if (c > best || (c == best && b - a == 1)) { single = (b - a == 1) ? 1 : 0; best = c; }
      wk = fmax(c - cf[0], 0.0);
      const double du = ub_weight(s, ucf, b) - ub_weight(s, ucf, a);
      scale[k] = du > 0 ? wk / du : 0.0;
    }
    double inc = wk;  // inclusive scan over the 1024 threads
    for (int o = 1; o < 32; o <<= 1) {
      const double y = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += y;
    }
    if (lane == 31) sm[w] = inc;
    __syncthreads();
    double wb = s_carry;
    for (int q = 0; q < w; ++q) wb += sm[q];
    if (k < K) S[k] = wb + inc - wk;
    __syncthreads();
    if (tid == 1023) s_carry = wb + inc;
    __syncthreads();
  }
  __shared__ int sm_single[32];
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int os = __shfl_xor_sync(0xffffffffu, single, o);
    if (ob > best || (ob == best && os)) { best = ob; single = os; }
  }
  if (lane == 0) { sm[w] = best; sm_single[w] = single; }
  __syncthreads();
  if (tid == 0) {
    for (int q = 1; q < 32; ++q)
      if (sm[q] > best || (sm[q] == best && sm_single[q])) { best = sm[q]; single = sm_single[q]; }
    const double total = s_carry;
    S[K] = total;
    const double prev = first ? 0.0 : ctl->best;
    const double b = first ? best : fmin(prev, best);
    ctl->best = b;
    ctl->total = total;
    ctl->tlo = total / (double)K;
    if (first) { ctl->stop = 0; ctl->tstar = 0; }
    // balanced well inside the bisection's tolerance, or the last step gained less than 0.3 %: nothing left to gain
    if (!(best - cf[0] > (1.0 + fmax(0.004, tol)) * (total / (double)K))) ctl->stop = 1;
    if (!first && !(best < 0.997 * prev)) ctl->stop = 1;
    // the costliest part is a single column: no partition can do better than that column alone -- the bound is the optimum
    if (single) ctl->stop = 1;
    // the step's greedy threshold on the rescaled weight predicted this bottleneck within 1 %: the weight model is consistent
    // with the exact costs, another step would cut at the same places
    if (!first && best - cf[0] <= 1.01 * ctl->tstar) ctl->stop = 1;
    out[0] = b;
    out[1] = ctl->stop ? 1.0 : 0.0;
  }
}

// grid point i = the last column boundary whose rescaled weight is at most i / UB_G of the total
__global__ void __launch_bounds__(256) k_ub_grid(const __grid_constant__ DevStream s, int is_float, int K, const int* __restrict__ spl,
                                                 const double* __restrict__ S, const double* __restrict__ scale, const UbCtl* __restrict__ ctl,
                                                 u32* __restrict__ gx, float* __restrict__ gw) {
  if (ctl->stop) return;
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i > UB_G) return;
  double cf[4];
  for (int t = 0; t < 4; ++t) cf[t] = is_float ? s.cf[t] : (double)s.ci[t];
  if (!(cf[1] + cf[2] + cf[3] > 0)) { cf[1] = 1; cf[2] = 0; cf[3] = 0; }
  const double total = S[K];
  const double target = total * ((double)i / (double)UB_G);
  int lo = 0, hi = K;  // largest k < K with S[k] <= target (k = K - 1 at the very end)
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (S[mid] <= target) lo = mid; else hi = mid;
  }
  const int k = lo;
  const u32 a = (u32)spl[k], b = (u32)spl[k + 1];
  const double ua = ub_weight(s, cf, a), sc = scale[k];
  u32 x = a;
  if (i == UB_G) x = s.n + 1;
  else if (sc > 0) {
    const double ut = ua + (target - S[k]) / sc;
    u32 l = a, h = b;  // largest x in [a, b] with U(x) <= ut
    while (l < h) {
      const u32 mid = l + ((h - l + 1) >> 1);
      if (ub_weight(s, cf, mid) <= ut) l = mid; else h = mid - 1;
    }
    x = l;
  }
  gx[i] = x;
  // rescaled weight at x: x lies in [a, b] of part k
  gw[i] = (float)(i == UB_G ? total : S[k] + sc * (ub_weight(s, cf, x) - ua));
}

// parametric search: candidate t cuts the grid greedily at threshold T_t (geometric ladder from the mean share to eight times
// the mean share: a column may outweigh the mean share by far); the smallest threshold that places every
// column in at most K parts gives the new partition
static constexpr int UB_CTA = 32;  // candidate thresholds per CTA: one warp per SM walks the grid out of its own shared-memory copy
__global__ void __launch_bounds__(UB_CTA) k_ub_greedy(int K, UbCtl* __restrict__ ctl, const float* __restrict__ gw_g, u32* __restrict__ cuts, int* __restrict__ first) {
  extern __shared__ float s_gw[];  // UB_G + 1
  if (ctl->stop) return;
  const int tid = threadIdx.x;
  for (int i = tid; i <= UB_G; i += UB_CTA) s_gw[i] = gw_g[i];
  __syncthreads();
  const int t = blockIdx.x * UB_CTA + tid;  // candidate index 0 .. UB_T - 1
  const float total = s_gw[UB_G];
  const double tlo = ctl->tlo;
  const float T = (float)(tlo * exp2(3.0 * (double)t / (double)(UB_T - 1)));
  const float w0 = total / (float)UB_G;
  u32* my = cuts + (size_t)t * (K + 1);
  int i = 0;
  bool ok = true;
  my[0] = 0;
  for (int k = 1; k <= K; ++k) {
    if (i < UB_G) {
      const float target = s_gw[i] + T;
      int lo = i, hi = UB_G;  // largest index with s_gw <= target
      const int g = min(UB_G, i + (int)(T / w0));
      if (s_gw[g] <= target) { lo = g; const int g2 = min(UB_G, g + 8); if (s_gw[g2] > target) hi = g2; }
      else { hi = g; const int g2 = max(i, g - 8); if (s_gw[g2] <= target) lo = g2; }
      while (lo < hi) {
        const int mid = lo + ((hi - lo + 1) >> 1);
        if (s_gw[mid] <= target) lo = mid; else hi = mid - 1;
      }
      // (grid points that share a column boundary carry the same weight: the search lands on the last of them)
      if (lo == i) { ok = false; break; }  // one step outweighs T
      i = lo;
    }
    my[k] = (u32)i;
  }
  if (ok && i == UB_G) atomicMin(first, t);
}
// the smallest threshold that placed every column gives the new partition (none: the partition stays)
__global__ void __launch_bounds__(1024) k_ub_apply(int K, UbCtl* __restrict__ ctl, const u32* __restrict__ gx, const u32* __restrict__ cuts, int* __restrict__ first,
                                                   int* __restrict__ spl) {
  if (ctl->stop) return;
  const int best = *first;
  __syncthreads();
  if (threadIdx.x == 0) {
    *first = UB_T;  // (armed for the next step)
    if (best < UB_T) ctl->tstar = ctl->tlo * exp2(3.0 * (double)best / (double)(UB_T - 1));
  }
  if (best >= UB_T) return;
  const u32* src = cuts + (size_t)best * (K + 1);
  for (int k = threadIdx.x; k <= K; k += 1024) spl[k] = (k == 0) ? 1 : (int)gx[src[k]];
}

// The same bound for the models probed through the dominance index: parts cut at equal shares of (columns + pins),
// their costs evaluated with K oracle queries.
template <class T>
__global__ void k_ub_index(const __grid_constant__ DevOracle o, int K, double* __restrict__ out) {
  __shared__ double sm[32];
  const u32 n1 = o.n + 1;
  const double N = (double)__ldg(o.pos + o.n), n = (double)o.n;
  auto weight = [&](u32 x) { return (double)(x - 1) * (N + 1) + (double)__ldg(o.pos + (x - 1)) * (n + 1); };  // x = 1..n+1
  const double total = weight(n1);
  auto cut = [&](int k) -> u32 {  // smallest x with weight(x) >= k / K of the total
    if (k <= 0) return 1u;
    if (k >= K) return n1;
    const double target = total * ((double)k / (double)K);
    u32 lo = 1, hi = n1;
    while (lo < hi) {
      const u32 mid = lo + ((hi - lo) >> 1);
      if (weight(mid) >= target) hi = mid; else lo = mid + 1;
    }
    return lo;
  };
  double best = 0;
  for (int k = threadIdx.x; k < K; k += blockDim.x) best = fmax(best, (double)dev_cost<T>(o, cut(k), cut(k + 1), (u32)k + 1u));
  for (int off = 16; off > 0; off >>= 1) best = fmax(best, __shfl_xor_sync(0xffffffffu, best, off));
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = best;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) best = fmax(best, sm[w]);
    out[0] = best;
  }
}

// ---- one bisection as a sequence of steps, so that the nodes of a round can be probed by different
//      ranks (the sharded solve, sharded.cu) ----
struct BisectRun {
  Oracle* f = nullptr;
  bool stream = false;
  i64 K = 0;
  double eps1 = 1;
  int P = 1;
  DBuf<BisectState> st;
  DBuf<int> hint_lo, hint_hi, best, ids;
  // per node of the round: 1-based split points ((K+2) each), result (0 = loop condition already false, 1 = infeasible,
  // 2 = feasible), threshold
  DBuf<int> node_spl, node_res;
  DBuf<double> node_c;
  DevStream ds{};
  bool done = false;
  double c_lo0 = 0, c_hi0 = 0, eps = 0;
  // speculation plan of the current round: slot t probes tree node h_ids[t] (heap index)
  BisectState h_st{};
  std::vector<int> h_ids, h_best;  // h_best: host copy of `best`, refreshed with every synchronising advance
  bool planned = false, adaptive = true;
  i64 speculated = 0;  // thresholds probed so far (this rank)
  double ub = 0;  // upper bound on the optimal bottleneck (0 = unknown)
};

// Prior over the optimal bottleneck c*: log-uniform over the initial bracket, mixed with a log-uniform bump just below
// the heuristic upper bound when one is known.  A tree node is reached by the walk iff c* lies in its (c_lo, c_hi].
struct PlanPrior {
  double c_lo0, c_hi0, ub;  // initial bracket, planner's upper bound (0 = none)
};
static double prior_mass(const PlanPrior& pr, double lo, double hi) {
  auto lu = [](double lo, double hi, double a, double b) {
    lo = std::max(lo, a);
    hi = std::min(hi, b);
    return (hi > lo && a > 0 && b > a) ? (std::log(hi) - std::log(lo)) / (std::log(b) - std::log(a)) : 0.0;
  };
  if (!(pr.c_lo0 > 0) || !(pr.c_hi0 > pr.c_lo0)) return hi - lo;
  if (!(pr.ub > pr.c_lo0)) return lu(lo, hi, pr.c_lo0, pr.c_hi0);
  // the bound is the bottleneck of an actual partition, so c* <= ub: no mass above it.  Most of the mass sits just
  // below the bound (on near-uniform matrices the bounding partition is within a percent of the optimum).
  const double top = std::min(pr.ub * (1 + 1e-9), pr.c_hi0);
  return 0.1 * lu(lo, hi, pr.c_lo0, top) + 0.3 * lu(lo, hi, std::max(pr.ub / 1.5, pr.c_lo0), top) +
         0.6 * lu(lo, hi, std::max(pr.ub / 1.03, pr.c_lo0), top);
}

// Chooses the P tree nodes of the next round (heap indices, -1 = unused slot): greedily those the sequential loop is
// most likely to visit (a node's probability is the prior mass of its bracket; a parent's bracket contains its
// children's, so the set is a subtree containing the root).  With a flat prior this is the complete tree in heap order.
// Pure host arithmetic: every rank computes the same plan from the same state.  The plan only decides what is probed
// speculatively -- the thresholds themselves and the walk are the reference's sequence.
void bisect_plan_nodes(double c_lo, double c_hi, double eps, int P, double c_lo0, double c_hi0, double ub, bool adaptive, int* ids_out) {
  int count = 0;
  if (!adaptive) {
    for (int t = 0; t < P; ++t) ids_out[count++] = t;
    return;
  }
  const double eps1 = 1 + eps;
  const PlanPrior pr{c_lo0, c_hi0, ub};
  struct Cand { double mass; int depth; int heap; double lo, hi; };
  auto worse = [](const Cand& a, const Cand& b) {
    if (a.mass != b.mass) return a.mass < b.mass;
    if (a.depth != b.depth) return a.depth > b.depth;
    return a.heap > b.heap;
  };
  std::priority_queue<Cand, std::vector<Cand>, decltype(worse)> pq(worse);
  pq.push({prior_mass(pr, c_lo, c_hi), 0, 0, c_lo, c_hi});
  while (!pq.empty() && count < P) {
    const Cand x = pq.top();
    pq.pop();
    if (!(x.lo * eps1 < x.hi)) continue;  // the loop stops here: nothing to probe
    ids_out[count++] = x.heap;
    if (x.depth + 1 > BS_MAX_DEPTH) continue;
    const double c = (x.lo + x.hi) / 2;
    pq.push({prior_mass(pr, x.lo, c), x.depth + 1, 2 * x.heap + 1, x.lo, c});  // feasible: c_hi = c
    pq.push({prior_mass(pr, c, x.hi), x.depth + 1, 2 * x.heap + 2, c, x.hi});  // infeasible: c_lo = c
  }
  while (count < P) ids_out[count++] = -1;  // unused slots (never matched by the walk)
}

static void plan_round(BisectRun& run) {
  const int P = run.P;
  run.h_ids.assign(P, -1);
  bisect_plan_nodes(run.h_st.c_lo, run.h_st.c_hi, run.eps, P, run.c_lo0, run.c_hi0, run.ub, run.adaptive, run.h_ids.data());
  CPB_CUDA(cudaMemcpyAsync(run.ids.get(), run.h_ids.data(), (size_t)P * sizeof(int), cudaMemcpyHostToDevice, ctx().stream));
  run.planned = true;
}

// DevStream view of the oracle's link stream
static void stream_view(Oracle& f, DevStream& ds) {
  const Matrix& A = *f.A;
  ds.prev = f.ls->prev.get();
  ds.colq = f.ls->colq.get();
  ds.P = f.ls->P;
  ds.Wt = (f.dev.kind == CPB_MODEL_MONOSYM) ? f.overpos.get() - 1 : A.pos.get() - 1;
  ds.Ne = (u32)f.ls->Ne;
  ds.n = (u32)A.n;
  ds.same_w = ds.Wt == ds.P;
  for (int t = 0; t < 4; ++t) { ds.cf[t] = f.dev.cf[t]; ds.ci[t] = f.dev.ci[t]; }
}

// planner's upper bound (see k_ub_splits, k_ub_prepare) into d_out[0]; d_out[1] = 1 when the bounding partition is balanced
// (or cannot be refined); asynchronous
struct UbWork {
  DBuf<int> spl;
  DBuf<u32> cnt;
  DBuf<double> S, scale;
  DBuf<UbCtl> ctl;
  unsigned slices = 1;
  int steps = 0;
};
static void launch_upper_bound(Oracle& f, const DevStream& ds, i64 K, double eps, int nodes, double* d_out, UbWork& w) {
  ProfScope pk("probe_plan_bound");
  w.spl.alloc(K + 1);
  w.cnt.alloc(K);
  CPB_LAUNCH(k_ub_splits, (unsigned)((K + 1 + 255) / 256), 256, 0, ds, f.dev.is_float, (int)K, w.spl.get(), w.cnt.get());
  w.slices = (unsigned)std::min<i64>(64, std::max<i64>(1, ((i64)ctx().sm_count * 8 + K - 1) / K));
  CPB_LAUNCH(k_ub_count, dim3(w.slices, (unsigned)K, 1), 256, 0, ds, w.spl.get(), w.cnt.get(), (const int*)nullptr);
  // (also for wide rounds: 60 thresholds -- four ranks -- did NOT cover R-MAT 24's loose bound in one round, measured)
  (void)nodes;
  w.steps = (K <= UB_KMAX && f.A->n >= 4 * K) ? env_int("CPB_UB_REFINE", 3) : 0;
  if (w.steps <= 0) {
    CPB_LAUNCH(k_ub_max, 1, 256, 0, ds, f.dev.is_float, (int)K, w.spl.get(), w.cnt.get(), d_out);
    return;
  }
  w.S.alloc(K + 1);
  w.scale.alloc(K);
  w.ctl.alloc(1);
  CPB_LAUNCH(k_ub_prepare, 1, 1024, 0, ds, f.dev.is_float, (int)K, w.spl.get(), w.cnt.get(), w.S.get(), w.scale.get(), w.ctl.get(), d_out, 1, eps / 4);
}
// refinement steps of the bounding partition (the host saw that it is not balanced); asynchronous
static void refine_upper_bound(Oracle& f, const DevStream& ds, i64 K, double eps, double* d_out, UbWork& w) {
  ProfScope pk("probe_plan_bound");
  static bool attr_set = false;
  if (!attr_set) {
    CPB_CUDA(cudaFuncSetAttribute(k_ub_greedy, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((UB_G + 1) * sizeof(float))));
    attr_set = true;
  }
  DBuf<u32> gx(UB_G + 1), cuts((size_t)UB_T * (K + 1));
  DBuf<float> gw(UB_G + 1);
  DBuf<int> first(1);
  const int armed = UB_T;
  CPB_CUDA(cudaMemcpyAsync(first.get(), &armed, sizeof(int), cudaMemcpyHostToDevice, ctx().stream));
  int* const stop = &w.ctl.get()->stop;
  for (int it = 0; it < w.steps; ++it) {
    CPB_LAUNCH(k_ub_grid, (UB_G + 256) / 256, 256, 0, ds, f.dev.is_float, (int)K, w.spl.get(), w.S.get(), w.scale.get(), w.ctl.get(), gx.get(), gw.get());
    CPB_LAUNCH(k_ub_greedy, UB_T / UB_CTA, UB_CTA, (UB_G + 1) * sizeof(float), (int)K, w.ctl.get(), gw.get(), cuts.get(), first.get());
    CPB_LAUNCH(k_ub_apply, 1, 1024, 0, (int)K, w.ctl.get(), gx.get(), cuts.get(), first.get(), w.spl.get());
    CPB_LAUNCH(k_ub_zero, (unsigned)((K + 255) / 256), 256, 0, w.cnt.get(), (int)K, stop);
    CPB_LAUNCH(k_ub_count, dim3(w.slices, (unsigned)K, 1), 256, 0, ds, w.spl.get(), w.cnt.get(), stop);
    CPB_LAUNCH(k_ub_prepare, 1, 1024, 0, ds, f.dev.is_float, (int)K, w.spl.get(), w.cnt.get(), w.S.get(), w.scale.get(), w.ctl.get(), d_out, 0, eps / 4);
    if (env_int("CPB_UB_DEBUG", 0)) {  // (measurements: the state after every step)
      UbCtl h{};
      CPB_CUDA(cudaMemcpyAsync(&h, w.ctl.get(), sizeof(h), cudaMemcpyDeviceToHost, ctx().stream));
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));
      std::fprintf(stderr, "[cpb ub] step %d: best %.0f, greedy threshold %.0f, mean share %.0f, stop %d\n", it + 1, h.best, h.tstar, h.tlo, h.stop);
    }
  }
}

// The device's part searches count the feasible samples of an INCREASING predicate.  The reference's windowed binary search
// (BisectCost...:22-39) is path dependent for a cost that shrinks as the part grows (a work model with a negative beta --
// bound_stripe accepts it, WorkCosts.jl:37-51), so such models are refused instead of answered differently (ADVICE r1).
static void require_monotone_cost(const Oracle& f) {
  if (f.mdl.kind == CPB_MODEL_COLBLOCK || f.mdl.kind == CPB_MODEL_BLOCK) return;  // (tabulated: checked by the bound)
  for (int t = 1; t <= 3; ++t)
    if (f.mdl.coef[t] < 0)
      throw Error(CPB_ERR_UNSUPPORTED, "bisection on the device needs a cost that grows with the part (beta >= 0); a shrinking cost makes the reference's "
                                       "windowed search path dependent");
}

// The leading probes of the sequential loop that the planner's bound settles (see bisect_begin): walks them with the loop's own
// expressions and returns the c_hi they leave and their number.  Pure host arithmetic (cpb_bisect_prewalk exposes it to the
// CPU tests).
void bisect_prewalk(double c_lo, double c_hi, double eps, double ub, double* c_hi_out, int* probes_out) {
  const double eps1 = 1 + eps;
  const double safe = ub * eps1 * eps1;
  int probes = 0;
  while (c_lo * eps1 < c_hi) {
    const double c = (c_lo + c_hi) / 2;
    if (!(c >= safe)) break;
    // (the argument needs an infeasible probe to end the loop.  bound_stripe's lower bound is not a bound for every model -- the
    //  envelope's (c_hi - alpha) / K can exceed the optimum, EnvelopeCosts.jl:30-42 -- and then the loop ends on the INITIAL c_lo
    //  with feasible probes only: the probe that would end the loop is its last feasible one and runs for real.  Found by
    //  tests/fuzz_parity.py, seed 41.)
    if (!(c_lo * eps1 < c)) break;
    c_hi = c;
    probes += 1;
  }
  *c_hi_out = c_hi;
  *probes_out = probes;
}

void BisectRunDelete::operator()(BisectRun* run) const { delete run; }

BisectRunPtr bisect_begin(Oracle& f, bool lazy, double eps, i64 K, int nodes) {
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  CPB_REQUIRE(f.dev.kind != CPB_MODEL_BLOCK, "bisection needs a random-access oracle");
  require_monotone_cost(f);
  const Matrix& A = *f.A;
  CPB_REQUIRE(A.n + 1 < ((i64)1 << 31) && K + 2 < ((i64)1 << 30), "problem too large for 32-bit split points");
  BisectRunPtr run(new BisectRun);
  run->f = &f;
  run->K = K;
  run->adaptive = env_int("CPB_BISECT_PLAN", 1) != 0;
  // Connectivity-type models stream the link array (no dominance index needed); the others walk the index.
  run->stream = (f.dev.kind == CPB_MODEL_CONNECTIVITY || f.dev.kind == CPB_MODEL_MONOSYM) && env_int("CPB_PROBE_STREAM", 1) != 0;
  if (run->stream) {
    // Everything the host needs before the first round -- the row-degree check of the link construction, nets(1, n+1)
    // or the over-pin total for bound_stripe, the planner's upper bound -- is produced without waiting and read back
    // with ONE synchronisation.
    const bool dia = f.dev.kind == CPB_MODEL_MONOSYM;
    if (!f.ls) {
      ProfScope prof("oracle_stripe");
      // (large patterns: check the row degree first -- a wasted gigabyte-sized segment allocation costs far more than
      //  the ~20 us round trip the deferred check saves)
      f.ls = build_link_stream(A, dia, /*defer_check=*/A.N < ((i64)1 << 25), false, /*as_pos=*/true);
    }
    trace_mark("links");
    const bool want_ub = run->adaptive && K >= 2 && K <= 65535 && A.n >= 1;  // (K is the y extent of the counting grid)
    DBuf<double> ub_out(2);
    UbWork ubw;
    double h_ub[2] = {0, 1};
    for (int attempt = 0; attempt < 2; ++attempt) {
      stream_view(f, run->ds);
      if (want_ub) launch_upper_bound(f, run->ds, K, eps, nodes, ub_out.get(), ubw);
      u32 info[2] = {0, 0}, n_over = 0;
      CPB_CUDA(cudaMemcpyAsync(info, f.ls->first_count.get(), sizeof(info), cudaMemcpyDeviceToHost, ctx().stream));
      if (dia) CPB_CUDA(cudaMemcpyAsync(&n_over, f.overpos.get() + A.n, sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
      if (want_ub) CPB_CUDA(cudaMemcpyAsync(h_ub, ub_out.get(), (ubw.steps > 0 ? 2 : 1) * sizeof(double), cudaMemcpyDeviceToHost, ctx().stream));
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));
      run->ub = h_ub[0];
      if (f.ls->speculative && !dia) A.max_row_deg = (i64)info[1];
      if (f.ls->speculative && info[1] > LT_MAX_DEG) {  // a heavy row: the row-segment kernels did nothing -> stable sort
        ProfScope prof("oracle_stripe");
        f.ls = build_link_stream(A, dia, false, /*force_sort=*/true, /*as_pos=*/true);
        continue;
      }
      trace_mark("plan_bound");
      f.ls->speculative = false;
      f.ls->h_first_count = info[0];
      if (dia) f.h_n_over = n_over;
      if (want_ub && ubw.steps > 0 && h_ub[1] == 0.0) {
        // the bounding partition is not balanced: refine it (a second, short round trip -- only where it can save a round)
        refine_upper_bound(f, run->ds, K, eps, ub_out.get(), ubw);
        CPB_CUDA(cudaMemcpyAsync(h_ub, ub_out.get(), sizeof(double), cudaMemcpyDeviceToHost, ctx().stream));
        CPB_CUDA(cudaStreamSynchronize(ctx().stream));
        run->ub = h_ub[0];
      }
      break;
    }
  } else {
    oracle_ensure_ranks(f);
    bool monotone = true;  // the bound is only meaningful for costs that grow with the part (beta >= 0)
    for (int t = 1; t <= 4; ++t) monotone = monotone && (f.mdl.coef[t] >= 0 || (f.mdl.kind == CPB_MODEL_MONOSYM && t == 4));
    if (run->adaptive && K >= 2 && A.n >= 1 && monotone && f.dev.kind != CPB_MODEL_COLBLOCK) {
      ProfScope pk("probe_plan_bound");
      DBuf<double> ub_out(1);
      if (f.dev.is_float) CPB_LAUNCH(k_ub_index<double>, 1, 256, 0, f.dev, (int)K, ub_out.get());
      else CPB_LAUNCH(k_ub_index<i64>, 1, 256, 0, f.dev, (int)K, ub_out.get());
      CPB_CUDA(cudaMemcpyAsync(&run->ub, ub_out.get(), sizeof(double), cudaMemcpyDeviceToHost, ctx().stream));
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));
    }
  }
  double bnd[2];
  oracle_bound(f, K, bnd);  // (c_lo, c_hi) ./ 1
  if (lazy) {
    // LazyBisect...:55-57 / :233-235: c_lo = max(c_lo, f(empty part k)) -- alpha for the affine models
    double a0 = f.mdl.coef[0];
    if (f.mdl.kind == CPB_MODEL_COLBLOCK) a0 = f.h_alpha_col[0];
    bnd[0] = std::max(bnd[0], a0);
  }
  if (!run->stream)
    // the rank descents are dependent random sector reads: make them L2 hits when the index fits
    for (RankStruct* rs : {f.net.get(), f.dianet.get(), f.selfnet.get(), f.selfpin.get()})
      if (rs && rs->wm.bytes() > 0 && rs->wm.bytes() <= ((size_t)64 << 20) && env_int("CPB_L2_PREFETCH", 1)) {
        const size_t bytes = rs->wm.bytes();
        const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>((bytes / 128 + 255) / 256, (size_t)ctx().sm_count * 8));
        CPB_LAUNCH(k_l2_prefetch, grid, 256, 0, (const char*)rs->wm.blocks.get(), bytes);
      }
  // the round's speculation tree: `nodes` slots, filled by plan_round
  run->P = std::min(std::max(nodes, 1), BS_MAX_NODES);
  run->eps1 = 1 + eps;
  const int P = run->P;
  run->st.alloc(1);
  run->ids.alloc(P);
  run->hint_lo.alloc(K + 2);
  run->hint_hi.alloc(K + 2);
  run->best.alloc(K + 2);
  run->h_best.assign(K + 2, 0);
  run->node_spl.alloc((size_t)P * (K + 2));
  run->node_res.alloc(P);
  run->node_c.alloc(P);
  run->node_spl.zero();
  BisectState h{};
  h.c_lo = bnd[0];
  h.c_hi = bnd[1];
  run->c_lo0 = h.c_lo; run->c_hi0 = h.c_hi; run->eps = eps;
  // The planner's bound settles the leading probes of the sequential loop without running them.  The bound is the
  // bottleneck of an actual partition, so the optimum is at most ub, and the greedy probe of a monotone cost succeeds at
  // every threshold that is at least the optimum: the loop's first thresholds c = (c_lo + c_hi) / 2 >= ub (1 + eps)^2 are
  // feasible for certain and only move c_hi (BisectCost...:53-55).  They are walked here, with the loop's own expressions,
  // so every later threshold is the reference's.  None of them can be the loop's LAST feasible probe -- whose split vector
  // is the result: if it were, the loop would have ended with c_lo (1 + eps) >= c_hi >= ub (1 + eps)^2, i.e. with an
  // infeasible (or initial) c_lo above ub, which no threshold below the optimum is.  On R-MAT scale 24 this skips 5 of 13
  // probes and the remaining 8 fit one round of 15 speculated thresholds instead of two.
  if (run->ub > 0 && eps >= 1e-12 && env_int("CPB_BISECT_PREWALK", 1) != 0) {
    int walked = 0;
    bisect_prewalk(h.c_lo, h.c_hi, eps, run->ub, &h.c_hi, &walked);
    h.probes += walked;
  }
  h.done = !(h.c_lo * run->eps1 < h.c_hi);
  run->done = h.done != 0;
  run->h_st = h;
  CPB_CUDA(cudaMemcpyAsync(run->st.get(), &run->h_st, sizeof(h), cudaMemcpyHostToDevice, ctx().stream));
  CPB_LAUNCH(k_bisect_init, 1, 256, 0, (int)K, (int)(A.n + 1), run->hint_lo.get(), run->hint_hi.get(), run->best.get());
  if (run->done) {  // no probe will run: the answer is the initial spl_hi = [1, n+1, ..., n+1] (BisectCost...:32-33)
    CPB_CUDA(cudaMemcpyAsync(run->h_best.data(), run->best.get(), (K + 2) * sizeof(int), cudaMemcpyDeviceToHost, ctx().stream));
    CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  }
  return run;
}

static unsigned long long* g_probe_dbg_host = nullptr;
static std::string probe_debug_string() {
  if (!g_probe_dbg_host || g_probe_dbg_host[0] == 0) return "";
  const unsigned long long w0 = g_probe_dbg_host[0], w1 = g_probe_dbg_host[1], w2 = g_probe_dbg_host[2];
  char buf[256];
  std::snprintf(buf, sizeof(buf), " [probe wait timed out: tag=%llu crank=%llu block=%llu tid=%llu a=%llu b=%llu c=%llu d=%llu]", (w0 >> 4) & 15, (w0 >> 8) & 15,
                (w0 >> 12) & 0xffff, (w0 >> 28) & 0xfff, w1 >> 32, w1 & 0xffffffffull, w2 >> 32, w2 & 0xffffffffull);
  return buf;
}
// the host-mapped record a timed-out wait leaves (see probe_wait_failed)
static void probe_debug_arm() {
  if (g_probe_dbg_host) return;
  unsigned long long* d = nullptr;
  CPB_CUDA(cudaHostAlloc((void**)&g_probe_dbg_host, 128, cudaHostAllocMapped));
  std::memset(g_probe_dbg_host, 0, 128);
  CPB_CUDA(cudaHostGetDevicePointer((void**)&d, g_probe_dbg_host, 0));
  CPB_CUDA(cudaMemcpyToSymbol(g_probe_dbg, &d, sizeof(d)));
}
static void check_probes(cudaError_t e) {
  if (e != cudaSuccess) throw Error(CPB_ERR_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e) + " in the bisection probes" + probe_debug_string());
}

// probes the nodes [node_lo, node_hi) of the current round's speculation tree
void bisect_probe(BisectRun& run, int node_lo, int node_hi) {
  node_lo = std::max(node_lo, 0);
  node_hi = std::min(node_hi, run.P);
  if (node_hi <= node_lo) return;
  Oracle& f = *run.f;
  const int K = (int)run.K;
  if (!run.planned) plan_round(run);
  for (int t = node_lo; t < node_hi; ++t) run.speculated += run.h_ids[t] >= 0;
  for (int base = node_lo; base < node_hi; base += (1 << BS_LOCAL_DEPTH)) {
    const int cnt = std::min(node_hi - base, 1 << BS_LOCAL_DEPTH);
    if (run.stream) {
      // algorithmic bytes of one fused pass over the links for the thresholds of this launch (SURVEY.md 8d, G4)
      ProfScope pk("k_probe_stream", (double)(f.ls->Ne + f.A->n + 1) * 4.0 + (double)cnt * (K + 1) * 8.0);
      probe_debug_arm();
      if (f.dev.is_float)
        CPB_LAUNCH(k_probe_stream<double>, cnt * BS_CLUSTER, SP_THREADS, 0, run.ds, K, run.eps1, run.st.get(), run.node_spl.get(), run.node_res.get(), run.node_c.get(), run.ids.get(), base);
      else
        CPB_LAUNCH(k_probe_stream<i64>, cnt * BS_CLUSTER, SP_THREADS, 0, run.ds, K, run.eps1, run.st.get(), run.node_spl.get(), run.node_res.get(), run.node_c.get(), run.ids.get(), base);
    } else if (f.dev.is_float) {
      CPB_LAUNCH(k_bisect_round<double>, cnt * BS_CLUSTER, BS_THREADS, 0, f.dev, K, run.eps1, run.st.get(), run.hint_lo.get(), run.hint_hi.get(), run.node_spl.get(), run.node_res.get(), run.node_c.get(), run.ids.get(), base);
    } else {
      CPB_LAUNCH(k_bisect_round<i64>, cnt * BS_CLUSTER, BS_THREADS, 0, f.dev, K, run.eps1, run.st.get(), run.hint_lo.get(), run.hint_hi.get(), run.node_spl.get(), run.node_res.get(), run.node_c.get(), run.ids.get(), base);
    }
  }
}

// walks the (complete) tree of the round; `sync` reads back whether the bisection has finished
bool bisect_advance(BisectRun& run, bool sync) {
  if (!run.planned) plan_round(run);  // (advance without a probe: the walk stops at the root)
  CPB_LAUNCH(k_bisect_advance, 1, 256, 0, (int)run.K, run.P, run.eps1, run.st.get(), run.hint_lo.get(), run.hint_hi.get(), run.best.get(),
             run.node_spl.get(), run.node_res.get(), run.node_c.get(), run.ids.get());
  if (sync) {
    check_probes(cudaMemcpyAsync(&run.h_st, run.st.get(), sizeof(BisectState), cudaMemcpyDeviceToHost, ctx().stream));
    check_probes(cudaMemcpyAsync(run.h_best.data(), run.best.get(), (run.K + 2) * sizeof(int), cudaMemcpyDeviceToHost, ctx().stream));
    check_probes(cudaStreamSynchronize(ctx().stream));
    run.done = run.h_st.done != 0;
    run.planned = false;  // the next round is planned from the new bracket
  }
  return run.done;
}

void bisect_node_buffers(BisectRun& run, int** res, double** c, int** spl, int* P) {
  *res = run.node_res.get(); *c = run.node_c.get(); *spl = run.node_spl.get(); *P = run.P;
}
bool bisect_is_done(BisectRun& run) { return run.done; }

static double g_bisect_stats[8] = {0, 0, 0, 0, 0, 0, 0, 0};
void bisect_stats(double out[8]) {
  for (int t = 0; t < 8; ++t) out[t] = g_bisect_stats[t];
}

void bisect_finish(const BisectRun& run, int64_t* h_spl_out) {
  CPB_REQUIRE(run.done, "bisection has not finished");
  const i64 K = run.K;
  g_bisect_stats[0] = run.h_st.rounds; g_bisect_stats[1] = run.h_st.probes; g_bisect_stats[2] = (double)run.speculated;
  g_bisect_stats[3] = run.c_lo0; g_bisect_stats[4] = run.c_hi0; g_bisect_stats[5] = run.ub;
  g_bisect_stats[6] = run.h_st.c_lo; g_bisect_stats[7] = run.h_st.c_hi;
  for (i64 k = 1; k <= K + 1; ++k) h_spl_out[k - 1] = run.h_best[k];  // read back by the last advance
}

#ifdef CPB_PROBE_TIMING
void probe_timing_dump() {
  unsigned long long t[16], n;
  cudaMemcpyFromSymbol(t, g_probe_t, sizeof(t));
  cudaMemcpyFromSymbol(&n, g_probe_n, sizeof(n));
  {
    unsigned long long nd[16][4];
    cudaMemcpyFromSymbol(nd, g_probe_node, sizeof(nd));
    for (int i = 0; i < 16; ++i)
      if (nd[i][3]) std::printf("probe_timing slot %2d: launches %llu, per launch: %.0f cycles, %.1f super-steps, %.1f parts, %.0f cycles/super-step\n", i, nd[i][3],
                                (double)nd[i][0] / nd[i][3], (double)nd[i][1] / nd[i][3], (double)nd[i][2] / nd[i][3], (double)nd[i][0] / std::max<unsigned long long>(nd[i][1], 1));
    unsigned long long z[16][4] = {{0}};
    cudaMemcpyToSymbol(g_probe_node, z, sizeof(z));
  }
  const char* names[11] = {"loads+flags", "syncthreads", "scan(warp0)", "push+exchange 1", "boundaries", "push+exchange 2", "top of the tile loop", "read exchange 2",
                           "loop exit + tile estimate", "part bookkeeping", "top of the part loop"};
  for (int i = 0; i < 11; ++i) std::printf("probe_timing %-22s %8.1f cycles/super-step\n", names[i], (double)t[i] / (double)std::max<unsigned long long>(n, 1));
  std::printf("probe_timing super-steps %llu\n", n);
  unsigned long long parts[4];
  cudaMemcpyFromSymbol(parts, g_probe_parts, sizeof(parts));
  std::printf("probe_timing parts slot0 %llu slot1 %llu slot2 %llu ; super-steps slot1 %llu\n", parts[0], parts[1], parts[2], parts[3]);
}
#endif

// how many 8-CTA probe clusters the device can keep resident at once (cluster placement is per GPC)
int probe_cluster_capacity(bool stream) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(BS_CLUSTER * 64, 1, 1);
  cfg.blockDim = dim3(stream ? SP_THREADS : BS_THREADS, 1, 1);
  cfg.dynamicSmemBytes = 0;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = BS_CLUSTER;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  if (stream) CPB_CUDA(cudaOccupancyMaxActiveClusters(&n, k_probe_stream<i64>, &cfg));
  else CPB_CUDA(cudaOccupancyMaxActiveClusters(&n, k_bisect_round<i64>, &cfg));
  return n;
}

// The checks of a BisectIndex solve; leaves the oracle's bound (c_lo, c_hi) in bnd.
static void bisect_index_prepare(Oracle& f, i64 K, double bnd[2]) {
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  CPB_REQUIRE(f.dev.kind != CPB_MODEL_BLOCK, "bisection needs a random-access oracle");
  const Matrix& A = *f.A;
  CPB_REQUIRE(A.n + 1 < ((i64)1 << 31) && K + 2 < ((i64)1 << 30), "problem too large for 32-bit split points");
  require_monotone_cost(f);
  oracle_ensure_ranks(f);
  oracle_bound(f, K, bnd);  // (c_lo, c_hi) ./ 1 -- also checks beta >= 0, which the monotone part searches need
}

// The checks of a Flip solve (method: CPB_SPLIT_FLIP_BISECT_COST, CPB_SPLIT_LAZY_FLIP_BISECT_COST or CPB_SPLIT_FLIP_BISECT_INDEX).
static void flip_prepare(Oracle& f, i64 K, double bnd[2]) {
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  CPB_REQUIRE(f.dev.kind == CPB_MODEL_SECCONN || f.dev.kind == CPB_MODEL_SECEDGE, "the Flip splitters on the device serve the (decreasing) secondary models");
  if (f.dev.kind == CPB_MODEL_SECCONN)
    CPB_REQUIRE(f.mdl.coef[3] <= f.mdl.coef[4], "Flip splitters need a cost that does not grow with the part (beta_local_net <= beta_remote_net)");
  else
    CPB_REQUIRE(f.mdl.coef[2] <= f.mdl.coef[3], "Flip splitters need a cost that does not grow with the part (beta_self_pin <= beta_cut_pin)");
  const Matrix& A = *f.A;
  CPB_REQUIRE(A.n + 1 < ((i64)1 << 31) && K + 2 < ((i64)1 << 30), "problem too large for 32-bit split points");
  CPB_REQUIRE(K == f.pi_K, "the secondary model's row partition must have K parts");
  oracle_ensure_ranks(f);
  oracle_bound(f, K, bnd);
}

// One problem of k_stripe_batch, checked exactly as the single solvers check it (their messages).
static StripeJob prepare_job(Oracle& f, int method, const double* eps, i64 K) {
  if (method != CPB_SPLIT_BISECT_INDEX && method != CPB_SPLIT_FLIP_BISECT_COST && method != CPB_SPLIT_LAZY_FLIP_BISECT_COST && method != CPB_SPLIT_FLIP_BISECT_INDEX)
    throw Error(CPB_ERR_UNSUPPORTED, "a batch takes the BisectIndex and Flip splitters only");
  const bool cost = method == CPB_SPLIT_FLIP_BISECT_COST || method == CPB_SPLIT_LAZY_FLIP_BISECT_COST;
  CPB_REQUIRE(eps || !cost, "eps is NULL but a FlipBisectCost method needs it");
  double bnd[2];
  if (method == CPB_SPLIT_BISECT_INDEX) bisect_index_prepare(f, K, bnd);
  else flip_prepare(f, K, bnd);
  StripeJob jb{};
  jb.method = method;
  jb.K = (int)K;
  jb.lazy = method == CPB_SPLIT_LAZY_FLIP_BISECT_COST;
  jb.c_lo = bnd[0];
  jb.c_hi = bnd[1];
  jb.eps1 = cost ? 1 + *eps : 1.0;
  return jb;
}

// Launches checked jobs (one launch per cost type) and copies the split vectors out.  The workspace holds, per problem, the
// vector the solve returns (spl_hi for BisectIndex and LazyFlipBisectCost, spl_lo for FlipBisectCost and FlipBisectIndex, as
// in the reference) in one contiguous region, read back with one copy, and its two other vectors behind it.  The vectors
// are 1-based: slot 0 of the returned one carries the problem's probe count.
static void run_jobs(i64 B, Oracle* const* f, std::vector<StripeJob>& jobs, int64_t* const* h_spl_out, int* h_probes) {
  std::vector<const Oracle*> distinct;
  std::vector<i64> res_off(B);
  i64 res_total = 0;
  for (i64 b = 0; b < B; ++b) {
    const auto it = std::find(distinct.begin(), distinct.end(), f[b]);
    jobs[b].oracle = (int)(it - distinct.begin());
    if (it == distinct.end()) distinct.push_back(f[b]);
    res_off[b] = res_total;
    res_total += jobs[b].K + 2;
  }
  // Int64 problems first, then Float64
  std::vector<StripeJob> sorted;
  i64 other = res_total, n_int = 0;
  for (int is_float = 0; is_float < 2; ++is_float)
    for (i64 b = 0; b < B; ++b) {
      if (f[b]->dev.is_float != is_float) continue;
      StripeJob jb = jobs[b];
      const i64 n = jb.K + 2;
      const bool keep_hi = jb.method == CPB_SPLIT_BISECT_INDEX || jb.lazy;
      jb.spl = other;
      (keep_hi ? jb.spl_lo : jb.spl_hi) = other + n;
      (keep_hi ? jb.spl_hi : jb.spl_lo) = res_off[b];
      jb.probes = res_off[b];
      other += 2 * n;
      sorted.push_back(jb);
      n_int += !is_float;
    }
  const size_t oracle_bytes = distinct.size() * sizeof(DevOracle);
  std::vector<char> table(oracle_bytes + B * sizeof(StripeJob));
  for (size_t i = 0; i < distinct.size(); ++i) std::memcpy(table.data() + i * sizeof(DevOracle), &distinct[i]->dev, sizeof(DevOracle));
  std::memcpy(table.data() + oracle_bytes, sorted.data(), B * sizeof(StripeJob));
  ProfScope prof("probe");
  DBuf<char> d_table(table.size());
  DBuf<int> ws((size_t)other);
  CPB_CUDA(cudaMemcpyAsync(d_table.get(), table.data(), table.size(), cudaMemcpyHostToDevice, ctx().stream));
  const DevOracle* d_or = reinterpret_cast<const DevOracle*>(d_table.get());
  const StripeJob* d_jobs = reinterpret_cast<const StripeJob*>(d_table.get() + oracle_bytes);
  if (n_int > 0) CPB_LAUNCH(k_stripe_batch<i64>, (unsigned)(n_int * BS_CLUSTER), BS_THREADS, 0, d_or, d_jobs, ws.get());
  if (B > n_int) CPB_LAUNCH(k_stripe_batch<double>, (unsigned)((B - n_int) * BS_CLUSTER), BS_THREADS, 0, d_or, d_jobs + n_int, ws.get());
  std::vector<int> h(res_total);
  CPB_CUDA(cudaMemcpyAsync(h.data(), ws.get(), res_total * sizeof(int), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  for (i64 b = 0; b < B; ++b) {
    const int* r = h.data() + res_off[b];
    for (i64 k = 1; k <= jobs[b].K + 1; ++k) h_spl_out[b][k - 1] = r[k];
    if (h_probes) h_probes[b] = r[0];
  }
}

// The single solves are batches of one: the batch kernel reads the oracle into shared memory, which measured faster than
// the kernel-parameter oracle of a one-problem kernel (DESIGN section 4).
void solve_bisect_index(Oracle& f, i64 K, int64_t* h_spl_out) {
  std::vector<StripeJob> jobs{prepare_job(f, CPB_SPLIT_BISECT_INDEX, nullptr, K)};
  Oracle* fp = &f;
  int hp = 0;
  run_jobs(1, &fp, jobs, &h_spl_out, &hp);
  g_bisect_stats[0] = 1; g_bisect_stats[1] = hp; g_bisect_stats[2] = hp;
  g_bisect_stats[3] = jobs[0].c_lo; g_bisect_stats[4] = jobs[0].c_hi; g_bisect_stats[5] = 0; g_bisect_stats[6] = 0; g_bisect_stats[7] = 0;
}

// method: CPB_SPLIT_FLIP_BISECT_COST, CPB_SPLIT_LAZY_FLIP_BISECT_COST or CPB_SPLIT_FLIP_BISECT_INDEX
void solve_flip(Oracle& f, int method, double eps, i64 K, int64_t* h_spl_out) {
  std::vector<StripeJob> jobs{prepare_job(f, method, &eps, K)};
  Oracle* fp = &f;
  run_jobs(1, &fp, jobs, &h_spl_out, nullptr);
}

// Every problem is checked first -- a failure names the problem, and nothing is launched or written.  cpb_bisect_stats is
// not updated.
void solve_stripe_batch(i64 B, Oracle* const* f, const int* method, const double* eps, const i64* K, int64_t* const* h_spl_out) {
  if (B <= 0) return;
  std::vector<StripeJob> jobs(B);
  for (i64 b = 0; b < B; ++b) {
    try {
      CPB_REQUIRE(f[b] && h_spl_out[b], "NULL argument");
      jobs[b] = prepare_job(*f[b], method[b], eps ? eps + b : nullptr, K[b]);
    } catch (const Error& e) {
      throw Error(e.code, "problem " + std::to_string(b) + ": " + e.what());
    }
  }
  run_jobs(B, f, jobs, h_spl_out, nullptr);
}

// how many stripe_batch clusters the device keeps resident at once
int stripe_batch_capacity() {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(BS_CLUSTER * 1024, 1, 1);
  cfg.blockDim = dim3(BS_THREADS, 1, 1);
  cfg.dynamicSmemBytes = 0;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = BS_CLUSTER;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  CPB_CUDA(cudaOccupancyMaxActiveClusters(&n, k_stripe_batch<i64>, &cfg));
  return n;
}

void solve_bisect(Oracle& f, bool lazy, double eps, i64 K, int64_t* h_spl_out) {
  const int depth = std::min(std::max(env_int("CPB_BISECT_DEPTH", BS_LOCAL_DEPTH), 1), BS_LOCAL_DEPTH);
  BisectRunPtr run = bisect_begin(f, lazy, eps, K, (1 << depth) - 1);
  trace_mark("begin");
  {
    ProfScope prof("probe");
    // The gap c_hi - c_lo halves with every probe and the loop stops once it is <= eps * c_lo, so the number
    // of rounds is bounded from the initial bounds: queue them all without host round trips (rounds past
    // the end find the state `done` and exit immediately), then read the state back once.
    if (!run->done && run->c_lo0 > 0 && run->eps > 0 && run->c_hi0 > run->c_lo0 && !run->adaptive && env_int("CPB_BISECT_QUEUE", 0)) {
      const double iters = std::ceil(std::log2((run->c_hi0 - run->c_lo0) / (run->eps * run->c_lo0))) + 2;
      const int rounds = (int)std::min(64.0, std::ceil(std::max(iters, 1.0) / depth) + 1);
      for (int r = 0; r < rounds; ++r) {
        bisect_probe(*run, 0, run->P);
        bisect_advance(*run, r + 1 == rounds);
      }
    }
    for (int guard = 0; guard < 4096 && !run->done; ++guard) {
      bisect_probe(*run, 0, run->P);
      trace_mark("probe");
      bisect_advance(*run, true);
      trace_mark("advance");
    }
    CPB_REQUIRE(run->done, "bisection did not terminate (eps too small for Float64?)");
  }
  bisect_finish(*run, h_spl_out);
  trace_mark("finish");
#ifdef CPB_PROBE_TIMING
  if (env_int("CPB_PROBE_TIMING_DUMP", 0)) probe_timing_dump();
#endif
}

}  // namespace cpb
