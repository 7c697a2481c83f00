// primitives.cu -- device-wide scan, stable radix sort and small index kernels (sm_100a).
#include <algorithm>
#include "primitives.cuh"

namespace cpb {

static constexpr unsigned FULL = 0xffffffffu;

int bits_for(u64 v) {
  int b = 1;
  while (b < 64 && (v >> b) != 0) ++b;
  return b;
}

// ------------------------------------------------------------------------------------ scan
static constexpr int SC_THREADS = 256;
static constexpr int SC_CHUNK = SC_THREADS * 4;  // items per block-scan step
static constexpr int SC_TILE = SC_CHUNK * 8;     // items per CTA

// exclusive scan of one value per thread across a 256-thread CTA; returns the exclusive prefix,
// `total` receives the CTA-wide sum.  smem: 8 words.
__device__ __forceinline__ u32 block_excl_scan_256(u32 x, u32* smem, u32& total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  u32 inc = x;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    u32 y = __shfl_up_sync(FULL, inc, o);
    if (lane >= o) inc += y;
  }
  if (lane == 31) smem[w] = inc;
  __syncthreads();
  u32 wbase = 0, tot = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    u32 s = smem[k];
    if (k < w) wbase += s;
    tot += s;
  }
  __syncthreads();
  total = tot;
  return wbase + inc - x;
}

__global__ void __launch_bounds__(SC_THREADS) k_scan_reduce(const u32* __restrict__ in, u32* __restrict__ sums, size_t n) {
  __shared__ u32 sm[8];
  const size_t b0 = (size_t)blockIdx.x * SC_TILE;
  const size_t b1 = min(n, b0 + (size_t)SC_TILE);
  u32 s = 0;
  for (size_t i = b0 + threadIdx.x; i < b1; i += SC_THREADS) s += in[i];
  u32 tot;
  block_excl_scan_256(s, sm, tot);
  if (threadIdx.x == 0) sums[blockIdx.x] = tot;
}

// scans [b0, b1) with starting carry; safe for in == out
__device__ __forceinline__ void scan_range(const u32* in, u32* out, size_t b0, size_t b1, u32 carry, u32* sm) {
  for (size_t c0 = b0; c0 < b1; c0 += SC_CHUNK) {
    const size_t i0 = c0 + (size_t)threadIdx.x * 4;
    u32 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = (i0 + k < b1) ? in[i0 + k] : 0u;
    u32 tsum = v[0] + v[1] + v[2] + v[3];
    u32 tot;
    u32 ex = block_excl_scan_256(tsum, sm, tot) + carry;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (i0 + k < b1) out[i0 + k] = ex;
      ex += v[k];
    }
    carry += tot;
  }
}

__global__ void __launch_bounds__(SC_THREADS) k_scan_small(const u32* in, u32* out, size_t n) {
  __shared__ u32 sm[8];
  scan_range(in, out, 0, n, 0u, sm);
}

__global__ void __launch_bounds__(SC_THREADS) k_scan_apply(const u32* in, u32* out, const u32* __restrict__ tile_off, size_t n) {
  __shared__ u32 sm[8];
  const size_t b0 = (size_t)blockIdx.x * SC_TILE;
  const size_t b1 = min(n, b0 + (size_t)SC_TILE);
  scan_range(in, out, b0, b1, tile_off[blockIdx.x], sm);
}

void exclusive_scan_u32(const u32* in, u32* out, size_t n) {
  if (n == 0) return;
  if (n <= (size_t)SC_TILE * 8) {
    CPB_LAUNCH(k_scan_small, 1, SC_THREADS, 0, in, out, n);
    return;
  }
  const size_t tiles = (n + SC_TILE - 1) / SC_TILE;
  DBuf<u32> sums(tiles);
  CPB_LAUNCH(k_scan_reduce, (unsigned)tiles, SC_THREADS, 0, in, sums.get(), n);
  exclusive_scan_u32(sums.get(), sums.get(), tiles);
  CPB_LAUNCH(k_scan_apply, (unsigned)tiles, SC_THREADS, 0, in, out, sums.get(), n);
}

// ------------------------------------------------------------------------------ radix sort
// Stable LSD radix sort, DB = 8 or 10 bits per pass (the width is chosen to minimise passes), tiles of 8192
// (key, payload) pairs:
//   k_rs_hist     per-tile digit histogram                      (digit-major table, then one scan)
//   k_rs_scatter  ranks every pair inside the tile (warp-level match_any rounds + per-digit walk over the
//                 16 warps), stages the tile in shared memory in sorted order and copies it out so that
//                 every digit run is written with coalesced stores.
static constexpr int RS_THREADS = 512;
static constexpr int RS_IPT = 16;
static constexpr int RS_TILE = RS_THREADS * RS_IPT;  // 8192 pairs per CTA, 512 per warp
static constexpr int RS_WARPS = RS_THREADS / 32;
static constexpr u32 RS_INVALID = 0xffffffffu;
template <int DB> constexpr size_t rs_smem() { return (size_t)RS_WARPS * (1 << DB) * 2 + (size_t)(1 << DB) * 4 * 2 + 64 + (size_t)RS_TILE * 8; }

// per-tile digit histogram, stored digit-major: hist[d * tiles + tile]
template <int DB>
__global__ void __launch_bounds__(256) k_rs_hist(const u32* __restrict__ keys, size_t n, int shift, u32* __restrict__ hist, u32 tiles) {
  constexpr int NB = 1 << DB;
  __shared__ u32 h[NB];
  for (int d = threadIdx.x; d < NB; d += 256) h[d] = 0;
  __syncthreads();
  const size_t base = (size_t)blockIdx.x * RS_TILE;
#pragma unroll 4
  for (int r = 0; r < RS_TILE / 256; ++r) {
    const size_t i = base + (size_t)r * 256 + threadIdx.x;
    if (i < n) atomicAdd(&h[(keys[i] >> shift) & (NB - 1)], 1u);
  }
  __syncthreads();
  for (int d = threadIdx.x; d < NB; d += 256) hist[(size_t)d * tiles + blockIdx.x] = h[d];
}

template <int DB>
__global__ void __launch_bounds__(RS_THREADS, 2) k_rs_scatter(const u32* __restrict__ keys_in, const u32* __restrict__ vals_in,
                                                              u32* __restrict__ keys_out, u32* __restrict__ vals_out, size_t n,
                                                              int shift, const u32* __restrict__ offs, u32 tiles, int iota_vals) {
  constexpr int NB = 1 << DB;
  constexpr int DPT = NB / 256;  // digits per thread of the first 256 threads (1 or 4)
  extern __shared__ __align__(16) unsigned char rs_smem_raw[];
  unsigned short* wh = reinterpret_cast<unsigned short*>(rs_smem_raw);              // [RS_WARPS][NB] counts, then tile-local bases
  u32* s_tot = reinterpret_cast<u32*>(rs_smem_raw + (size_t)RS_WARPS * NB * 2);     // [NB] tile-local base of every digit
  u32* s_gb = s_tot + NB;                                                           // [NB] global base - local base
  u32* s_wsum = s_gb + NB;                                                          // [8] warp totals of the digit scan
  u32* s_keys = s_wsum + 16;                                                        // [RS_TILE]
  u32* s_vals = s_keys + RS_TILE;                                                   // [RS_TILE]
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  for (int i = tid; i < RS_WARPS * NB; i += RS_THREADS) wh[i] = 0;
  __syncthreads();
  const size_t tbase = (size_t)blockIdx.x * RS_TILE;
  const size_t base = tbase + (size_t)w * (32 * RS_IPT);
  const u32 tile_n = (u32)min((size_t)RS_TILE, n - tbase);
  u32 key[RS_IPT], val[RS_IPT], rnk[RS_IPT];
#pragma unroll
  for (int r = 0; r < RS_IPT; ++r) {
    const size_t i = base + (size_t)r * 32 + lane;
    const bool ok = i < n;
    key[r] = ok ? keys_in[i] : 0u;
    val[r] = ok ? (iota_vals ? (u32)i : vals_in[i]) : 0u;
  }
  const unsigned lt = (1u << lane) - 1u;
#pragma unroll
  for (int r = 0; r < RS_IPT; ++r) {
    const size_t i = base + (size_t)r * 32 + lane;
    const u32 d = (i < n) ? ((key[r] >> shift) & (NB - 1)) : RS_INVALID;
    const unsigned m = __match_any_sync(FULL, d);
    const int leader = __ffs(m) - 1;
    u32 old = 0;
    if (d != RS_INVALID && lane == leader) {
      old = wh[w * NB + d];
      wh[w * NB + d] = (unsigned short)(old + __popc(m));
    }
    __syncwarp();
    old = __shfl_sync(FULL, old, leader);
    rnk[r] = old + (u32)__popc(m & lt);
  }
  __syncthreads();
  // per digit: exclusive walk over the warps (thread t < 256 owns digits t*DPT .. t*DPT+DPT-1), then an
  // exclusive scan of the digit totals
  u32 dtot[DPT];
  u32 tsum = 0;
  if (tid < 256) {
#pragma unroll
    for (int e = 0; e < DPT; ++e) {
      const int d = tid * DPT + e;
      u32 run = 0;
#pragma unroll 4
      for (int k = 0; k < RS_WARPS; ++k) {
        const u32 t = wh[k * NB + d];
        wh[k * NB + d] = (unsigned short)run;
        run += t;
      }
      dtot[e] = run;
      tsum += run;
    }
  }
  u32 inc = tsum;
  if (tid < 256) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const u32 y = __shfl_up_sync(FULL, inc, o);
      if (lane >= o) inc += y;
    }
    if (lane == 31) s_wsum[w] = inc;
  }
  __syncthreads();
  if (tid < 256) {
    u32 wb = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k)
      if (k < w) wb += s_wsum[k];
    u32 run = wb + inc - tsum;
#pragma unroll
    for (int e = 0; e < DPT; ++e) {
      const int d = tid * DPT + e;
      s_tot[d] = run;
      s_gb[d] = offs[(size_t)d * tiles + blockIdx.x] - run;
      run += dtot[e];
    }
  }
  __syncthreads();
  // stage the tile in sorted order
#pragma unroll
  for (int r = 0; r < RS_IPT; ++r) {
    const size_t i = base + (size_t)r * 32 + lane;
    if (i < n) {
      const u32 d = (key[r] >> shift) & (NB - 1);
      const u32 p = s_tot[d] + wh[w * NB + d] + rnk[r];
      s_keys[p] = key[r];
      s_vals[p] = val[r];
    }
  }
  __syncthreads();
  // coalesced copy-out: consecutive staged positions of one digit go to consecutive addresses
#pragma unroll
  for (int r = 0; r < RS_IPT; ++r) {
    const u32 p = (u32)r * RS_THREADS + tid;
    if (p < tile_n) {
      const u32 k = s_keys[p];
      const u32 dst = s_gb[(k >> shift) & (NB - 1)] + p;
      keys_out[dst] = k;
      vals_out[dst] = s_vals[p];
    }
  }
}

template <int DB>
static int radix_sort_passes(u32* keys, u32* vals, u32* keys_tmp, u32* vals_tmp, size_t n, int passes, bool iota_payload, const u32* first_keys) {
  constexpr int NB = 1 << DB;
  static bool attr_set = false;
  if (!attr_set) {
    CPB_CUDA(cudaFuncSetAttribute(k_rs_scatter<DB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rs_smem<DB>()));
    attr_set = true;
  }
  const u32 tiles = (u32)((n + RS_TILE - 1) / RS_TILE);
  DBuf<u32> hist((size_t)NB * tiles);
  int which = 0;
  for (int pass = 0; pass < passes; ++pass) {
    const int shift = pass * DB;
    const u32* ki = which ? keys_tmp : keys;
    if (pass == 0 && first_keys) ki = first_keys;  // read-only source of the first pass (saves a copy into `keys`)
    u32* vi = which ? vals_tmp : vals;
    u32* ko = which ? keys : keys_tmp;
    u32* vo = which ? vals : vals_tmp;
    {
      ProfScope pk("k_rs_hist", (double)n * 4.0);
      CPB_LAUNCH(k_rs_hist<DB>, tiles, 256, 0, ki, n, shift, hist.get(), tiles);
    }
    {
      ProfScope pk("rs_scan", (double)NB * tiles * 8.0);
      exclusive_scan_u32(hist.get(), hist.get(), (size_t)NB * tiles);
    }
    {
      ProfScope pk("k_rs_scatter", (double)n * 16.0);  // read + write one (key, payload) pair per element
      CPB_LAUNCH(k_rs_scatter<DB>, tiles, RS_THREADS, rs_smem<DB>(), ki, vi, ko, vo, n, shift, hist.get(), tiles, (pass == 0 && iota_payload) ? 1 : 0);
    }
    which ^= 1;
  }
  return which;
}

// Stable sort of (key, payload) by the low `bits` bits of key.  iota_payload: the payload is the element
// index, generated on the fly in the first pass (vals need not be initialised).  10-bit digits are used when
// they save a pass (17..20 and 25..30 key bits).
static int radix_sort_impl(u32* keys, u32* vals, u32* keys_tmp, u32* vals_tmp, size_t n, int bits, bool iota_payload, const u32* first_keys) {
  if (n == 0) return 0;
  const int p8 = (bits + 7) / 8, p10 = (bits + 9) / 10;
  if (p10 < p8) return radix_sort_passes<10>(keys, vals, keys_tmp, vals_tmp, n, p10, iota_payload, first_keys);
  return radix_sort_passes<8>(keys, vals, keys_tmp, vals_tmp, n, p8, iota_payload, first_keys);
}

int radix_sort_pairs(u32* keys, u32* vals, u32* keys_tmp, u32* vals_tmp, size_t n, int bits) {
  return radix_sort_impl(keys, vals, keys_tmp, vals_tmp, n, bits, false, nullptr);
}

int radix_sort_pairs_iota(const u32* keys_src, u32* keys, u32* vals, u32* keys_tmp, u32* vals_tmp, size_t n, int bits) {
  return radix_sort_impl(keys, vals, keys_tmp, vals_tmp, n, bits, true, keys_src);
}

// ------------------------------------------------------------------------------ small kernels
__global__ void k_narrow_minus1(const i64* __restrict__ src, u32* __restrict__ dst, size_t n, i64 lo, i64 hi, u32* flags) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  bool bad = false;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const i64 v = src[i];
    bad |= (v < lo) | (v > hi);
    dst[i] = (u32)(v - 1);
  }
  if (__any_sync(FULL, bad) && (threadIdx.x & 31) == 0) atomicOr(flags, 1u);
}
__global__ void k_narrow32_minus1(const int* __restrict__ src, u32* __restrict__ dst, size_t n, i64 lo, i64 hi, u32* flags) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  bool bad = false;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const i64 v = src[i];
    bad |= (v < lo) | (v > hi);
    dst[i] = (u32)(v - 1);
  }
  if (__any_sync(FULL, bad) && (threadIdx.x & 31) == 0) atomicOr(flags, 1u);
}
void narrow32_minus1(const int* src, u32* dst, size_t n, i64 lo, i64 hi, u32* flags) {
  if (n == 0) return;
  const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)ctx().sm_count * 16);
  CPB_LAUNCH(k_narrow32_minus1, grid, 256, 0, src, dst, n, lo, hi, flags);
}
void narrow_minus1(const i64* src, u32* dst, size_t n, i64 lo, i64 hi, u32* flags) {
  if (n == 0) return;
  const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)ctx().sm_count * 16);
  CPB_LAUNCH(k_narrow_minus1, grid, 256, 0, src, dst, n, lo, hi, flags);
}

__global__ void k_dec_check_u32(u32* v, size_t n, i64 lo, i64 hi, u32* flags) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  bool bad = false;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const i64 x = (i64)v[i];
    bad |= (x < lo) | (x > hi);
    v[i] = (u32)(x - 1);
  }
  if (__any_sync(FULL, bad) && (threadIdx.x & 31) == 0) atomicOr(flags, 1u);
}
void dec_check_u32(u32* v, size_t n, i64 lo, i64 hi, u32* flags) {
  if (n == 0) return;
  const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)ctx().sm_count * 16);
  CPB_LAUNCH(k_dec_check_u32, grid, 256, 0, v, n, lo, hi, flags);
}

__global__ void k_check_monotone(const u32* __restrict__ pos, size_t n, u32* flags) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  bool bad = false;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i + 1 < n; i += stride) bad |= pos[i] > pos[i + 1];
  if (__any_sync(FULL, bad) && (threadIdx.x & 31) == 0) atomicOr(flags, 2u);
}
void check_monotone(const u32* pos, size_t n, u32* flags) {
  if (n < 2) return;
  const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)ctx().sm_count * 16);
  CPB_LAUNCH(k_check_monotone, grid, 256, 0, pos, n, flags);
}

__global__ void k_iota(u32* dst, size_t n) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = (u32)i;
}
void iota_u32(u32* dst, size_t n) {
  if (n == 0) return;
  const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)ctx().sm_count * 16);
  CPB_LAUNCH(k_iota, grid, 256, 0, dst, n);
}

// colidx[q] = largest j with pos[j] <= q.  A CTA owns 2048 consecutive nonzeros: a cooperative 256-ary search (three rounds
// for a million columns) finds the column of its first nonzero, every column that starts inside the tile marks its first
// nonzero with its number (a run of empty columns shares one offset: the largest number wins), and a running maximum over
// the tile turns the marks into the column of every nonzero -- ~20 instructions per nonzero instead of a binary search each.
static constexpr int EX_TILE = 2048;
static constexpr int EX_PER = EX_TILE / 256;  // consecutive nonzeros per thread
__global__ void __launch_bounds__(256) k_expand_columns(const u32* __restrict__ pos, u32 ncol, u32* __restrict__ colidx, size_t N) {
  __shared__ __align__(16) u32 s_head[EX_TILE];
  __shared__ u32 s_wmax[8];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const size_t q0 = (size_t)blockIdx.x * EX_TILE;
#pragma unroll
  for (int k = 0; k < EX_PER; ++k) s_head[tid * EX_PER + k] = 0;
  // c_lo = largest j in [0, ncol) with pos[j] <= q0   (pos[0] = 0 <= q0 < N = pos[ncol])
  u32 lo = 0, hi = ncol;
  while (hi - lo > 1) {
    const u32 step = (hi - lo + 255) / 256;
    const u64 idx = (u64)lo + (u64)(tid + 1) * step;
    const bool ok = idx < hi && __ldg(pos + idx) <= q0;
    const u32 cnt = (u32)__syncthreads_count(ok);  // pos is monotone: the probes that hold form a prefix
    const u32 nlo = lo + cnt * step;
    hi = min(hi, nlo + step);
    lo = nlo;
  }
  const u32 c_lo = lo;
  __syncthreads();
  // columns after c_lo start behind q0; those that start inside the tile leave their mark
  for (u64 c = (u64)c_lo + 1 + tid; c < ncol; c += 256) {
    const size_t p = __ldg(pos + c);
    if (p >= q0 + EX_TILE) break;
    atomicMax(&s_head[p - q0], (u32)c);
  }
  __syncthreads();
  u32 v[EX_PER];
  u32 run = 0;
#pragma unroll
  for (int k = 0; k < EX_PER; ++k) {
    run = max(run, s_head[tid * EX_PER + k]);
    v[k] = run;
  }
  u32 inc = run;  // inclusive running maximum across the threads
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u32 y = __shfl_up_sync(FULL, inc, o);
    if (lane >= o) inc = max(inc, y);
  }
  if (lane == 31) s_wmax[w] = inc;
  __syncthreads();
  u32 before = c_lo;  // maximum over everything left of this thread
#pragma unroll
  for (int k = 0; k < 8; ++k)
    if (k < w) before = max(before, s_wmax[k]);
  const u32 left = __shfl_up_sync(FULL, inc, 1);
  if (lane > 0) before = max(before, left);
  const size_t base = q0 + (size_t)tid * EX_PER;
  if (base + EX_PER <= N) {
    uint4* dst = reinterpret_cast<uint4*>(colidx + base);
    dst[0] = make_uint4(max(v[0], before), max(v[1], before), max(v[2], before), max(v[3], before));
    dst[1] = make_uint4(max(v[4], before), max(v[5], before), max(v[6], before), max(v[7], before));
  } else {
#pragma unroll
    for (int k = 0; k < EX_PER; ++k)
      if (base + k < N) colidx[base + k] = max(v[k], before);
  }
}
void expand_columns(const u32* pos, u32 ncol, u32* colidx, size_t N) {
  if (N == 0) return;
  const u32 tiles = (u32)((N + EX_TILE - 1) / EX_TILE);
  CPB_LAUNCH(k_expand_columns, tiles, 256, 0, pos, ncol, colidx, N);
}

__global__ void k_segment_starts(const u32* __restrict__ keys, size_t n, u32* __restrict__ P, u32 domain) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p <= n; p += stride) {
    const i64 lo = (p == 0) ? 0 : (i64)keys[p - 1] + 1;
    const i64 hi = (p == n) ? (i64)domain : (i64)keys[p];
    for (i64 x = lo; x <= hi; ++x) P[x] = (u32)p;
  }
}
void segment_starts(const u32* sorted_keys, size_t n, u32* P, u32 domain) {
  const unsigned grid = (unsigned)std::min<size_t>((n + 1 + 255) / 256, (size_t)ctx().sm_count * 16);
  CPB_LAUNCH(k_segment_starts, grid, 256, 0, sorted_keys, n, P, domain);
}

__global__ void k_widen_plus(const u32* __restrict__ src, i64* __restrict__ dst, size_t n, i64 add) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = (i64)src[i] + add;
}
void widen_plus(const u32* src, i64* dst, size_t n, i64 add) {
  if (n == 0) return;
  const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)ctx().sm_count * 16);
  CPB_LAUNCH(k_widen_plus, grid, 256, 0, src, dst, n, add);
}

}  // namespace cpb
