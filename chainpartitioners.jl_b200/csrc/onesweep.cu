// onesweep.cu -- stable LSD radix sort of packed (key << 32 | payload) pairs with ONE read and ONE write of the pairs per
// 8-bit pass (sm_100a), and the link construction that sits on top of it (links.cu, sharded.cu).
//
// The digit histograms of ALL passes come from one sweep over the keys (k_os_hist), and a tile learns how many equal
// digits precede it from its predecessors' published counts (chained scan with decoupled look-back: every tile publishes
// its per-digit count as soon as it is known, then the inclusive prefix), so no pass reads the keys twice:
//   k_os_pass<MODE>   MODE 0: first pass, pairs formed on the fly from a u32 key array (payload = element index)
//                     MODE 1: pair -> pair
//                     MODE 2: the pairs arrive sorted by (row, position); the pass forms every nonzero's link from its left
//                             neighbour while loading and partitions (link << 32 | position) by windows of the position
//                             (so that the final scatter of the links stays inside L2, links.cu)
// Tiles take their number from an atomic counter, so a tile's predecessors have always started (forward progress of the
// look-back does not depend on the hardware's block scheduling order).
#include "onesweep.cuh"

namespace cpb {

static constexpr unsigned FULL = 0xffffffffu;
static constexpr int OS_THREADS = 256;
static constexpr int OS_IPT = 16;
static constexpr int OS_WARPS = OS_THREADS / 32;
static constexpr int OS_TILE = OS_THREADS * OS_IPT;  // 4096 pairs per CTA
// look-back state word: 0 = not yet published, count + 1 = the tile's own count (<= OS_TILE + 1), OS_INC | prefix = the
// inclusive prefix (< 2^31: every index the library accepts)
static constexpr u32 OS_INC = 1u << 31, OS_VAL = OS_INC - 1u;
static constexpr int OS_LOOKBACK = 4;  // predecessors inspected per round trip

// digit histograms of up to four 8-bit passes in one sweep over the keys: ghist[pass * 256 + digit]
__global__ void __launch_bounds__(256) k_os_hist(const u32* __restrict__ keys, size_t n, int passes, u32* __restrict__ ghist) {
  __shared__ u32 h[4 * 256];
  for (int i = threadIdx.x; i < 4 * 256; i += 256) h[i] = 0;
  __syncthreads();
  const size_t stride = (size_t)gridDim.x * 256 * 4;
  for (size_t i = ((size_t)blockIdx.x * 256 + threadIdx.x) * 4; i < n; i += stride) {
    u32 k[4];
    int cnt = 4;
    if (i + 4 <= n && (reinterpret_cast<size_t>(keys + i) & 15) == 0) {
      const uint4 v = *reinterpret_cast<const uint4*>(keys + i);
      k[0] = v.x; k[1] = v.y; k[2] = v.z; k[3] = v.w;
    } else {
      cnt = (int)min((size_t)4, n - i);
      for (int e = 0; e < cnt; ++e) k[e] = keys[i + e];
    }
    for (int e = 0; e < cnt; ++e)
      for (int p = 0; p < passes; ++p) atomicAdd(&h[p * 256 + ((k[e] >> (8 * p)) & 255u)], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < passes * 256; i += 256)
    if (h[i]) atomicAdd(&ghist[i], h[i]);
}

__device__ __forceinline__ u32 ld_state(const u32* p) { return *reinterpret_cast<const volatile u32*>(p); }
__device__ __forceinline__ void st_state(u32* p, u32 v) { *reinterpret_cast<volatile u32*>(p) = v; }

// exclusive scan of one value per thread over the 256 threads of the CTA; sm: 8 words
__device__ __forceinline__ u32 os_block_scan(u32 x, u32* sm) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  u32 inc = x;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u32 y = __shfl_up_sync(FULL, inc, o);
    if (lane >= o) inc += y;
  }
  if (lane == 31) sm[w] = inc;
  __syncthreads();
  u32 wb = 0;
#pragma unroll
  for (int k = 0; k < OS_WARPS; ++k)
    if (k < w) wb += sm[k];
  __syncthreads();
  return wb + inc - x;
}

struct OsLinkArgs {
  const u32* colidx;  // column of every position (links as columns) or unused (as_pos)
  int as_pos;         // link = 1 + position of the left neighbour (else 1 + its column)
  u32 q_off;          // added to position-valued links (sharded construction: the block's first position)
  u32* first_count;   // += number of links equal to 0
  u32* last_local;    // optional: last_local[row] = q_off + 1 + last position of the row
};

// One tile of one pass.  FULLT: the tile holds OS_TILE pairs (no bounds checks).
template <int MODE, bool FULLT>
__device__ __forceinline__ void os_tile_body(const u32* __restrict__ keys32, const u64* __restrict__ in, u64* __restrict__ out, size_t n, int dshift,
                                             u32 dstart, u32* __restrict__ state, const OsLinkArgs& la, u32 tile, u32 hot, u64* s_pair, u32 (*s_mask)[256], u32 (*s_cur)[256],
                                             u32* s_gbase, u32* s_scan) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const size_t tbase = (size_t)tile * OS_TILE;
  const size_t base = tbase + (size_t)w * (32 * OS_IPT);
  const u32 tile_n = FULLT ? (u32)OS_TILE : (u32)(n - tbase);
  const u32 wn = FULLT ? 32u * OS_IPT : (u32)min((size_t)(32 * OS_IPT), n > base ? n - base : (size_t)0);  // pairs of this warp
#define OS_OK(r) (FULLT || (u32)((r) * 32 + lane) < wn)

  u64 pr[OS_IPT];
  if (MODE == 0) {
#pragma unroll
    for (int r = 0; r < OS_IPT; ++r) {
      const size_t i = base + (size_t)r * 32 + lane;
      pr[r] = OS_OK(r) ? (((u64)keys32[i] << 32) | (u64)(u32)i) : 0ull;
    }
  } else {
#pragma unroll
    for (int r = 0; r < OS_IPT; ++r) pr[r] = OS_OK(r) ? in[base + (size_t)r * 32 + lane] : 0ull;
  }
  if (MODE == 2) {
    // pr[] = (row, position) in sorted order: the left neighbour of the same row gives the link
    u64 carry = ~0ull;  // the pair left of this warp's first one (a row index never equals 0xffffffff)
    if (lane == 0 && base > 0 && wn > 0) carry = in[base - 1];
    u32 firsts = 0;
#pragma unroll
    for (int r = 0; r < OS_IPT; ++r) {
      const u64 cur = pr[r];
      u64 up = __shfl_up_sync(FULL, cur, 1);
      if (lane == 0) up = carry;
      carry = __shfl_sync(FULL, cur, 31);
      if (OS_OK(r)) {
        const size_t i = base + (size_t)r * 32 + lane;
        const bool same = (u32)(up >> 32) == (u32)(cur >> 32);
        const u32 qp = (u32)up;
        u32 link = 0;
        if (same) link = la.as_pos ? la.q_off + qp + 1u : __ldg(la.colidx + qp) + 1u;
        firsts += link == 0u;
        if (la.last_local) {
          if (!same && i > 0) la.last_local[(u32)(up >> 32)] = la.q_off + qp + 1u;  // the left neighbour closes its row
          if (i + 1 == n) la.last_local[(u32)(cur >> 32)] = la.q_off + (u32)cur + 1u;
        }
        pr[r] = ((u64)link << 32) | (u64)(u32)cur;
      }
    }
    firsts = __reduce_add_sync(FULL, firsts);
    if (lane == 0 && firsts && la.first_count) atomicAdd(la.first_count, firsts);
  }

  // rank inside the warp: the lanes holding the same digit in a round form a group; the group reads the warp's count of the
  // digit so far, its first lane adds the group's size.  Two ways to find the group (measured on B200: tools/ubench/,
  // profiles/r02_session2.md section 2): MATCH.ANY costs ~2 cycles per DISTINCT value on the SM's one address-divergence unit (61
  // cycles for random 8-bit digits, 1.7 ms per pass at 2.6e8 pairs; cheaper for skewed digits); through shared memory
  // -- every lane ORs its bit into the (warp, digit) mask word and reads it back, the first lane clears it -- costs
  // ~10 wavefronts per round for random digits (0.5 ms per pass) but lanes on the same word serialise (skewed digits).
  // `hot` != 0 (the pass's most frequent digit holds more than 1/16 of the pairs): MATCH.ANY; else shared memory.
  // (ranks inside the warp fit 10 bits: two per register)
  const unsigned lt = (1u << lane) - 1u;
  u32 rk2[OS_IPT / 2];
  if (hot) {
#pragma unroll
    for (int r = 0; r < OS_IPT; ++r) {
      const u32 d = (u32)(pr[r] >> dshift) & 255u;
      const unsigned m = __match_any_sync(FULL, OS_OK(r) ? d : 0xffffffffu);
      u32 cur = 0;
      if (OS_OK(r)) cur = s_cur[w][d];
      __syncwarp();
      if (OS_OK(r) && (m & lt) == 0u) s_cur[w][d] = cur + (u32)__popc(m);
      __syncwarp();
      const u32 rank = cur + (u32)__popc(m & lt);
      if (r & 1) rk2[r >> 1] |= rank << 16; else rk2[r >> 1] = rank;
    }
  } else {
#pragma unroll
    for (int r = 0; r < OS_IPT; ++r) {
      const u32 d = (u32)(pr[r] >> dshift) & 255u;
      if (OS_OK(r)) atomicOr(&s_mask[w][d], 1u << lane);
      __syncwarp();
      u32 m = 0, cur = 0;
      if (OS_OK(r)) {
        m = s_mask[w][d];
        cur = s_cur[w][d];
      }
      __syncwarp();
      if (OS_OK(r) && (m & lt) == 0u) {
        s_mask[w][d] = 0u;
        s_cur[w][d] = cur + (u32)__popc(m);
      }
      __syncwarp();
      const u32 rank = cur + (u32)__popc(m & lt);
      if (r & 1) rk2[r >> 1] |= rank << 16; else rk2[r >> 1] = rank;
    }
  }
  __syncthreads();
  // digit `tid`: counts of the warps -> tile total, published at once
  u32 total = 0;
#pragma unroll
  for (int k = 0; k < OS_WARPS; ++k) total += s_cur[k][tid];
  u32* const my_state = state + (size_t)tile * 256 + tid;
  st_state(my_state, tile == 0 ? (OS_INC | total) : total + 1u);
  const u32 lbase = os_block_scan(total, s_scan);  // first staged slot of the digit
  {
    u32 run = lbase;
#pragma unroll
    for (int k = 0; k < OS_WARPS; ++k) {
      const u32 c = s_cur[k][tid];
      s_cur[k][tid] = run;  // first slot of warp k's share of the digit
      run += c;
    }
  }
  // decoupled look-back for digit `tid`: sum the predecessors' counts until one of them carries an inclusive prefix
  u32 excl = 0;
  if (tile > 0) {
    long long t = (long long)tile - 1;
    bool done = false;
    const long long t_start = clock64();
    while (!done) {
      u32 v[OS_LOOKBACK];
#pragma unroll
      for (int j = 0; j < OS_LOOKBACK; ++j) v[j] = (t - j >= 0) ? ld_state(state + (size_t)(t - j) * 256 + tid) : OS_INC;
#pragma unroll
      for (int j = 0; j < OS_LOOKBACK; ++j) {
        if (done) break;
        while (v[j] == 0u) {
          v[j] = ld_state(state + (size_t)(t - j) * 256 + tid);
          if (clock64() - t_start > (4ll << 30)) __trap();  // (a predecessor never published: fail loudly instead of hanging)
        }
        if (v[j] & OS_INC) {
          excl += v[j] & OS_VAL;
          done = true;
        } else {
          excl += v[j] - 1u;
        }
      }
      t -= OS_LOOKBACK;
    }
    st_state(my_state, OS_INC | (excl + total));
  }
  s_gbase[tid] = dstart + excl - lbase;
  __syncthreads();

#pragma unroll
  for (int r = 0; r < OS_IPT; ++r) {
    const u32 d = (u32)(pr[r] >> dshift) & 255u;
    if (OS_OK(r)) s_pair[s_cur[w][d] + ((r & 1) ? (rk2[r >> 1] >> 16) : (rk2[r >> 1] & 0xffffu))] = pr[r];
  }
  __syncthreads();
  // copy-out: consecutive slots of one digit go to consecutive addresses
#pragma unroll
  for (int r = 0; r < OS_IPT; ++r) {
    const u32 p = (u32)r * OS_THREADS + tid;
    if (FULLT || p < tile_n) {
      const u64 v = s_pair[p];
      out[s_gbase[(u32)(v >> dshift) & 255u] + p] = v;
    }
  }
#undef OS_OK
}

template <int MODE>
__global__ void __launch_bounds__(OS_THREADS, 3)
k_os_pass(const u32* __restrict__ keys32, const u64* __restrict__ in, u64* __restrict__ out, size_t n, int dshift, const u32* __restrict__ ghist,
          u32* __restrict__ state, u32* __restrict__ counter, OsLinkArgs la) {
  extern __shared__ __align__(16) u64 s_pair[];  // OS_TILE staged pairs
  __shared__ u32 s_mask[OS_WARPS][256];           // per warp and digit: lanes holding the digit in the current round
  __shared__ u32 s_cur[OS_WARPS][256];            // per warp and digit: count so far -> first slot of the warp's share of the digit
  __shared__ u32 s_hot;
  __shared__ u32 s_gbase[256];                    // global index of a digit's first slot minus the slot
  __shared__ u32 s_scan[OS_WARPS];
  __shared__ u32 s_tile;
  const int tid = threadIdx.x;
  if (tid == 0) s_tile = atomicAdd(counter, 1u);
#pragma unroll
  for (int k = 0; k < OS_WARPS; ++k) { s_mask[k][tid] = 0u; s_cur[k][tid] = 0u; }
  // where the digit `tid` starts in the output
  u32 dstart;
  if (MODE == 2) {
    dstart = (u32)min((unsigned long long)n, (unsigned long long)tid << dshift);
  } else {
    const u32 g = ghist[tid];
    dstart = os_block_scan(g, s_scan);
    // is the pass's most frequent digit heavy (more than 1/16 of the pairs)?
    const u32 best = __reduce_max_sync(FULL, g);
    if ((tid & 31) == 0) s_scan[tid >> 5] = best;
    __syncthreads();
    if (tid == 0) {
      u32 b = 0;
      for (int k = 0; k < OS_WARPS; ++k) b = max(b, s_scan[k]);
      s_hot = ((unsigned long long)b * 16ull > (unsigned long long)n) ? 1u : 0u;
    }
  }
  if (MODE == 2 && tid == 0) s_hot = 0u;  // (windows of the position: near-uniform digits)
  __syncthreads();
  const u32 tile = s_tile;
  const u32 hot = s_hot;
  if ((size_t)(tile + 1) * OS_TILE <= n) os_tile_body<MODE, true>(keys32, in, out, n, dshift, dstart, state, la, tile, hot, s_pair, s_mask, s_cur, s_gbase, s_scan);
  else os_tile_body<MODE, false>(keys32, in, out, n, dshift, dstart, state, la, tile, hot, s_pair, s_mask, s_cur, s_gbase, s_scan);
}

static size_t os_tiles(size_t n) { return (n + OS_TILE - 1) / OS_TILE; }

struct OsWork {
  DBuf<u32> ghist, state, counters;
  size_t tiles = 0;
  int used = 0;  // passes run so far (each takes its own counter and state block)
  void init(size_t n, int total_passes) {
    tiles = os_tiles(n);
    ghist.alloc(4 * 256);
    ghist.zero();
    counters.alloc((size_t)total_passes);
    counters.zero();
    state.alloc(tiles * 256 * (size_t)total_passes);
    state.zero();
  }
  u32* next_state() { return state.get() + (size_t)used * tiles * 256; }
  u32* next_counter() { return counters.get() + used; }
};

template <int MODE> static void os_launch(OsWork& wk, const u32* keys32, const u64* in, u64* out, size_t n, int dshift, const u32* ghist, OsLinkArgs la) {
  static bool attr_set = false;
  if (!attr_set) {
    CPB_CUDA(cudaFuncSetAttribute(k_os_pass<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(OS_TILE * sizeof(u64))));
    attr_set = true;
  }
  CPB_LAUNCH(k_os_pass<MODE>, (unsigned)wk.tiles, OS_THREADS, OS_TILE * sizeof(u64), keys32, in, out, n, dshift, ghist, wk.next_state(), wk.next_counter(), la);
  wk.used += 1;
}

static u64* os_sort_passes(OsWork& wk, const u32* keys, size_t n, int passes, u64* a, u64* b) {
  {
    ProfScope pk("k_os_hist", (double)n * 4.0);
    const unsigned grid = (unsigned)std::min<size_t>((n + 1023) / 1024, (size_t)ctx().sm_count * 8);
    CPB_LAUNCH(k_os_hist, grid, 256, 0, keys, n, passes, wk.ghist.get());
  }
  u64* src = nullptr;
  u64* dst = a;
  const OsLinkArgs none{nullptr, 1, 0u, nullptr, nullptr};
  for (int p = 0; p < passes; ++p) {
    ProfScope pk("k_os_pass", (double)n * (p == 0 ? 12.0 : 16.0));
    if (p == 0) os_launch<0>(wk, keys, nullptr, dst, n, 32, wk.ghist.get(), none);
    else os_launch<1>(wk, nullptr, src, dst, n, 32 + 8 * p, wk.ghist.get() + 256 * p, none);
    src = dst;
    dst = (dst == a) ? b : a;
  }
  return src;
}

u64* onesweep_sort_iota(const u32* keys, size_t n, int bits, u64* a, u64* b) {
  CPB_REQUIRE(n > 0 && n < ((size_t)1 << 31), "onesweep: 0 < n < 2^31 pairs");
  const int passes = std::max(1, (bits + 7) / 8);
  OsWork wk;
  wk.init(n, passes);
  return os_sort_passes(wk, keys, n, passes, a, b);
}

// prev[position] = link for pairs (link << 32 | position)
__global__ void __launch_bounds__(256) k_os_scatter(const u64* __restrict__ pairs, size_t n, u32* __restrict__ prev) {
  const size_t i0 = ((size_t)blockIdx.x * 256 + threadIdx.x) * 2;
  if (i0 + 2 <= n) {
    const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(pairs + i0);
    prev[(u32)v.x] = (u32)(v.x >> 32);
    prev[(u32)v.y] = (u32)(v.y >> 32);
  } else if (i0 < n) {
    const u64 v = pairs[i0];
    prev[(u32)v] = (u32)(v >> 32);
  }
}

// links straight from the sorted (row, position) pairs (small inputs: the link array fits L2, no window pass)
__global__ void __launch_bounds__(256) k_os_link_scatter(const u64* __restrict__ sorted, size_t n, OsLinkArgs la, u32* __restrict__ prev) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  u32 firsts = 0;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += stride) {
    const u64 cur = sorted[p];
    const u64 up = p ? sorted[p - 1] : ~0ull;
    const bool same = (u32)(up >> 32) == (u32)(cur >> 32);
    const u32 qp = (u32)up;
    u32 link = 0;
    if (same) link = la.as_pos ? la.q_off + qp + 1u : __ldg(la.colidx + qp) + 1u;
    firsts += link == 0u;
    if (la.last_local) {
      if (!same && p > 0) la.last_local[(u32)(up >> 32)] = la.q_off + qp + 1u;
      if (p + 1 == n) la.last_local[(u32)(cur >> 32)] = la.q_off + (u32)cur + 1u;
    }
    prev[(u32)cur] = link;
  }
  firsts = __reduce_add_sync(FULL, firsts);
  if ((threadIdx.x & 31) == 0 && firsts && la.first_count) atomicAdd(la.first_count, firsts);
}

u64* onesweep_links(const u32* row, size_t N, int row_bits, const u32* colidx, bool as_pos, u32 q_off, u32* prev, u32* first_count, u32* last_local,
                    size_t window_min, u64* a, u64* b) {
  CPB_REQUIRE(N > 0 && N < ((size_t)1 << 31), "onesweep: 0 < N < 2^31 pairs");
  const int passes = std::max(1, (row_bits + 7) / 8);
  const bool windowed = window_min > 0 && N >= window_min;
  OsWork wk;
  wk.init(N, passes + (windowed ? 1 : 0));
  u64* sorted = os_sort_passes(wk, row, N, passes, a, b);
  const OsLinkArgs la{colidx, as_pos ? 1 : 0, q_off, first_count, last_local};
  ProfScope pk("k_link_prev", (double)N * 12.0);
  if (windowed) {
    // the link array does not fit L2, and a scatter in row order touches one HBM sector per 4-byte link (10.9 ms at
    // N = 2.6e8 on B200): one more pass groups (link, position) by 2^shift-position windows of `prev`, then the scatter
    // of a window stays in L2
    u64* other = (sorted == a) ? b : a;
    const int shift = std::max(0, bits_for(N - 1) - 8);
    os_launch<2>(wk, nullptr, sorted, other, N, shift, nullptr, la);
    CPB_LAUNCH(k_os_scatter, (unsigned)((N + 511) / 512), 256, 0, other, N, prev);
  } else {
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>((N + 255) / 256, (size_t)ctx().sm_count * 32));
    CPB_LAUNCH(k_os_link_scatter, grid, 256, 0, sorted, N, la, prev);
  }
  return sorted;
}

}  // namespace cpb
