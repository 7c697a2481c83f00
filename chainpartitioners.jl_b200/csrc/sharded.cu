// sharded.cu -- ONE stripe solve over several GPUs (one process per GPU), behind the C ABI with a library-owned NCCL
// communicator (SURVEY.md section 8b "Multi-GPU", 8e; BASELINE.json north_star: "column blocks of the oracle-construction
// sweep, candidate-threshold sets of the bisection ... NCCL over NVLink carries only ...").
//
//   * link construction (LazyBisectCostBottleneckSplitter.jl:156-192 builds cch[] = previous column of every nonzero with a
//     per-row "last seen" array): every rank owns a contiguous block of the CSC positions, [r * cnt, (r + 1) * cnt), and
//     uploads only that block of rowval.  It sorts its block by row (the transpose order of the block) -- the previous
//     nonzero of a row inside the block is the left neighbour in the row run.  For the first nonzero of a row inside a
//     block the predecessor lies in an earlier block: the per-row "last position seen" array (m * 4 bytes) travels down
//     the ranks once (rank r receives the running array from r - 1, fixes its run heads, merges its own last positions,
//     sends on), exactly the reference's hst[] carried across column blocks.  One in-place all-gather then gives every
//     rank the whole link array (N * 4 bytes) for the probes.  The monotonized symmetric model streams the links of A + I:
//     the same construction on each rank's block of A + I positions (see "A + I" below), gathered by per-rank broadcasts.
//   * adjointpattern of a sharded matrix (the alternation's second solve runs on the transpose): see below.
//   * bisection: the speculation tree of a round holds world x 15 thresholds; rank r probes slots [15 r, 15 (r + 1)) and
//     the per-slot results (feasible?, threshold, split vector) are all-gathered; every rank walks the same tree, so all
//     ranks end with the same state and the same split vector -- the reference's threshold sequence, hence its result.
//
// NCCL is loaded with dlopen at cpb_comm_init (no link-time dependency: the library loads on hosts without NCCL).
#include <dlfcn.h>
#include <nccl.h>
#include <chrono>
#include <vector>
#include "engine.cuh"
#include "primitives.cuh"
#include "onesweep.cuh"

namespace cpb {

struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
void host_pool_share(int ranks);  // hostpack.cpp
static NcclApi g_nccl;
static ncclComm_t g_comm = nullptr;
static int g_rank = 0, g_world = 1;
static double g_shard_stats[16] = {0};

#define CPB_NCCL(expr)                                                                                                              \
  do {                                                                                                                              \
    ncclResult_t _r = (expr);                                                                                                       \
    if (_r != ncclSuccess)                                                                                                          \
      throw ::cpb::Error(CPB_ERR_CUDA, std::string("NCCL error: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(_r) : "?") + " at " + __FILE__ + ":" + std::to_string(__LINE__)); \
  } while (0)

static void load_nccl() {
  if (g_nccl.lib) return;
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);  // the copy this process already holds (e.g. the host framework's)
  const char* env = std::getenv("CPB_NCCL_LIB");
  if (!h && env) h = dlopen(env, RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) throw Error(CPB_ERR_UNSUPPORTED, std::string("libnccl.so.2 not found (set CPB_NCCL_LIB): ") + dlerror());
  auto sym = [&](const char* name) {
    void* p = dlsym(h, name);
    if (!p) throw Error(CPB_ERR_UNSUPPORTED, std::string("NCCL symbol missing: ") + name);
    return p;
  };
  g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))sym("ncclGetUniqueId");
  g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))sym("ncclCommInitRank");
  g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))sym("ncclCommDestroy");
  g_nccl.AllGather = (decltype(g_nccl.AllGather))sym("ncclAllGather");
  g_nccl.AllReduce = (decltype(g_nccl.AllReduce))sym("ncclAllReduce");
  g_nccl.Broadcast = (decltype(g_nccl.Broadcast))sym("ncclBroadcast");
  g_nccl.Send = (decltype(g_nccl.Send))sym("ncclSend");
  g_nccl.Recv = (decltype(g_nccl.Recv))sym("ncclRecv");
  g_nccl.GroupStart = (decltype(g_nccl.GroupStart))sym("ncclGroupStart");
  g_nccl.GroupEnd = (decltype(g_nccl.GroupEnd))sym("ncclGroupEnd");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))sym("ncclGetErrorString");
  g_nccl.lib = h;
}

void comm_unique_id(char out[128]) {
  load_nccl();
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  CPB_NCCL(g_nccl.GetUniqueId(&id));
  std::memcpy(out, &id, 128);
}

void comm_init(const char id_bytes[128], int rank, int world) {
  CPB_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bad rank / world size");
  CPB_REQUIRE(world <= 16, "at most 16 ranks (the speculation tree of a round holds 255 thresholds)");
  load_nccl();
  if (g_comm) { g_nccl.CommDestroy(g_comm); g_comm = nullptr; }
  ncclUniqueId id;
  std::memcpy(&id, id_bytes, 128);
  CPB_NCCL(g_nccl.CommInitRank(&g_comm, world, id, rank));
  g_rank = rank;
  g_world = world;
  host_pool_share(world);  // the ranks of one box share its cores: each upload pool takes its share
}

void comm_destroy() {
  if (g_comm && g_nccl.CommDestroy) {
    cudaStreamSynchronize(ctx().stream);
    g_nccl.CommDestroy(g_comm);
  }
  g_comm = nullptr;
  g_rank = 0;
  g_world = 1;
}

void comm_info(int* rank, int* world) {
  if (rank) *rank = g_rank;
  if (world) *world = g_world;
}

// The element block of a rank: [r * cnt, min(N, (r + 1) * cnt)) with cnt = ceil(N / world) rounded up to 4 elements
// (equal counts make the link all-gather a plain in-place ncclAllGather; the tail falls into the padding of the array).
void shard_range(i64 N, int rank, int world, i64* cnt_out, i64* lo_out, i64* hi_out) {
  i64 cnt = (N + world - 1) / world;
  cnt = (cnt + 3) / 4 * 4;
  if (cnt_out) *cnt_out = cnt;
  if (lo_out) *lo_out = std::min<i64>(N, (i64)rank * cnt);
  if (hi_out) *hi_out = std::min<i64>(N, (i64)(rank + 1) * cnt);
}

struct ShardedMatrix {
  Matrix M;           // pos complete; row EMPTY (the pattern's rows live in row_blk, this rank's block only)
  DBuf<u32> row_blk;  // rows of the CSC positions [q_lo, q_hi)
  i64 cnt = 0, q_lo = 0, q_hi = 0;
  int rank = 0, world = 1;
};

static unsigned grid_for(size_t n) { return (unsigned)std::max<size_t>(1, std::min<size_t>((n + 255) / 256, (size_t)ctx().sm_count * 32)); }

// sorted (row, local position) pairs of the block -> link of every pair in sorted order (run heads: 0 for now) and the
// last position (+1) of every row of the block
__global__ void k_shard_link_values(const u32* __restrict__ sk, const u32* __restrict__ sq, size_t cnt, u32 q_lo, u32* __restrict__ lv,
                                    u32* __restrict__ last_local) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < cnt; p += stride) {
    const u32 r = sk[p];
    const bool head = p == 0 || sk[p - 1] != r;
    const bool tail = p + 1 == cnt || sk[p + 1] != r;
    lv[p] = head ? 0u : q_lo + sq[p - 1] + 1u;
    if (tail) last_local[r] = q_lo + sq[p] + 1u;
  }
}
__global__ void k_shard_scatter(const u32* __restrict__ sq, const u32* __restrict__ lv, size_t cnt, u32* __restrict__ prev_blk) {
  const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < cnt) prev_blk[sq[p]] = lv[p];
}
// run heads: the predecessor is the last position of the row in the earlier blocks (carry), none if the carry is 0
__global__ void k_shard_heads(const u32* __restrict__ sk, const u32* __restrict__ sq, size_t cnt, const u32* __restrict__ carry,
                              u32* __restrict__ prev_blk, u32* __restrict__ first_count) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  u32 firsts = 0;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < cnt; p += stride) {
    const u32 r = sk[p];
    if (p == 0 || sk[p - 1] != r) {
      const u32 c = carry ? carry[r] : 0u;
      if (c) prev_blk[sq[p]] = c;
      firsts += c == 0u;
    }
  }
  firsts = __reduce_add_sync(0xffffffffu, firsts);
  if ((threadIdx.x & 31) == 0 && firsts) atomicAdd(first_count, firsts);
}
__global__ void k_carry_merge(const u32* __restrict__ last_local, const u32* __restrict__ carry_in, u32* __restrict__ out, size_t m) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) {
    const u32 l = last_local[i];
    out[i] = l ? l : (carry_in ? carry_in[i] : 0u);
  }
}

// carry[i] = the last position (+1) of row i in the blocks of the ranks below `rank`: the nearest non-empty entry
__global__ void k_carry_pick(const u32* __restrict__ all, size_t m, int rank, u32* __restrict__ carry) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) {
    u32 c = 0;
    for (int r = rank - 1; r >= 0 && c == 0; --r) c = all[(size_t)r * m + i];
    carry[i] = c;
  }
}

static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// run heads of the packed (row << 32 | local position) pairs: as k_shard_heads
__global__ void k_shard_heads_pairs(const u64* __restrict__ sorted, size_t cnt, const u32* __restrict__ carry, u32* __restrict__ prev_blk,
                                    u32* __restrict__ first_count) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  u32 firsts = 0;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < cnt; p += stride) {
    const u64 cur = sorted[p];
    const u32 r = (u32)(cur >> 32);
    if (p == 0 || (u32)(sorted[p - 1] >> 32) != r) {
      const u32 c = carry ? carry[r] : 0u;
      if (c) prev_blk[(u32)cur] = c;
      firsts += c == 0u;
    }
  }
  firsts = __reduce_add_sync(0xffffffffu, firsts);
  if ((threadIdx.x & 31) == 0 && firsts) atomicAdd(first_count, firsts);
}

// one block's share of the construction: sort, in-block links, last positions
struct BlockWork {
  DBuf<u32> k0, v0, k1, v1, last_local;
  DBuf<u64> pa, pb;      // one-sweep form: packed pairs
  u64* sorted = nullptr;  // (row << 32 | local position), sorted
  u32 *sk = nullptr, *sq = nullptr;
  size_t cntL = 0;
};
static void block_local_links(const u32* row_blk, size_t cntL, u32 q_lo, size_t m, u32* prev_full, BlockWork& w) {
  ProfScope pk("shard_links_local", (double)(2 * cntL) * 4.0);
  w.cntL = cntL;
  w.last_local.alloc(std::max<size_t>(m, 1));
  CPB_CUDA(cudaMemsetAsync(w.last_local.get(), 0, std::max<size_t>(m, 1) * sizeof(u32), ctx().stream));
  if (!cntL) return;
  const char* wmin_env = std::getenv("CPB_WINDOWED_SCATTER_MIN");
  const size_t wmin = wmin_env ? (size_t)std::atoll(wmin_env) : ((size_t)1 << 25);
  u32* const prev_blk = prev_full + q_lo;
  const char* os_env = std::getenv("CPB_ONESWEEP");
  if (onesweep_supported(cntL) && !(os_env && os_env[0] == '0')) {
    // one-sweep radix passes on packed pairs (onesweep.cu): in-block links (run heads: 0 for now) and last positions
    w.pa.alloc(cntL);
    w.pb.alloc(cntL);
    w.sorted = onesweep_links(row_blk, cntL, bits_for(m ? m - 1 : 0), nullptr, /*as_pos=*/true, q_lo, prev_blk, nullptr, w.last_local.get(), wmin, w.pa.get(),
                              w.pb.get());
    return;
  }
  w.k0.alloc(cntL); w.v0.alloc(cntL); w.k1.alloc(cntL); w.v1.alloc(cntL);
  const int which = radix_sort_pairs_iota(row_blk, w.k0.get(), w.v0.get(), w.k1.get(), w.v1.get(), cntL, bits_for(m ? m - 1 : 0));
  w.sk = which ? w.k1.get() : w.k0.get();
  w.sq = which ? w.v1.get() : w.v0.get();
  u32* const other_k = which ? w.k0.get() : w.k1.get();
  u32* const other_v = which ? w.v0.get() : w.v1.get();
  CPB_LAUNCH(k_shard_link_values, grid_for(cntL), 256, 0, w.sk, w.sq, cntL, q_lo, other_k, w.last_local.get());
  if (wmin > 0 && cntL >= wmin) {
    // the block's links no longer fit L2: group the (position, link) pairs by windows of the link array first (see links.cu)
    DBuf<u32> pk2(cntL);
    const int shift = std::max(0, bits_for(cntL - 1) - 8);
    radix_partition_pass(w.sq, other_k, pk2.get(), other_v, cntL, shift);
    CPB_LAUNCH(k_shard_scatter, (unsigned)((cntL + 255) / 256), 256, 0, pk2.get(), other_v, cntL, prev_blk);
  } else {
    CPB_LAUNCH(k_shard_scatter, (unsigned)((cntL + 255) / 256), 256, 0, w.sq, other_k, cntL, prev_blk);
  }
}
static void block_heads(const BlockWork& w, const u32* carry_in, u32 q_lo, u32* prev_full, u32* first_count) {
  if (!w.cntL) return;
  if (w.sorted) CPB_LAUNCH(k_shard_heads_pairs, grid_for(w.cntL), 256, 0, w.sorted, w.cntL, carry_in, prev_full + q_lo, first_count);
  else CPB_LAUNCH(k_shard_heads, grid_for(w.cntL), 256, 0, w.sk, w.sq, w.cntL, carry_in, prev_full + q_lo, first_count);
}

// ---- A + I: the monotonized symmetric model streams the links of A + I (links.cu, build_link_stream(dia = true)) ----------
// A virtual diagonal (j, j) is appended to every column j that lacks one (SparseColorArrays.jl:87-91).  Position q of A moves
// to img(q) = q + addscan[c(q)] in A + I, c(q) the column holding q.  Rank r's block of A + I is [img(q_lo), img(q_hi)) with
// img(N) = N2 and rank 0 starting at 0: a virtual diagonal goes with the last real element of its column, and the diagonals
// of leading empty columns go to rank 0.  The blocks are contiguous, ordered and cover [0, N2); every rank computes all.

// the column holding element q < pos[n]: the largest c < n with pos[c] <= q (a non-empty column)
__device__ __forceinline__ u32 column_of(const u32* __restrict__ pos, u32 n, u32 q) {
  u32 lo = 0, hi = n - 1;
  while (lo < hi) {
    const u32 mid = lo + ((hi - lo + 1) >> 1);
    if (__ldg(pos + mid) <= q) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// present[j] = 1 if the part of column j inside the block [q_lo, q_hi) holds row j (the binary search of k_diag_missing on
// that part; rows ascend inside a column).  Flags of several blocks combine with MAX.
__global__ void k_shard_diag_present(const u32* __restrict__ pos, const u32* __restrict__ row_blk, u32 n, u32 q_lo, u32 q_hi,
                                     unsigned char* __restrict__ present) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) {
    u32 lo = max(__ldg(pos + j), q_lo), hi = min(__ldg(pos + j + 1), q_hi);
    if (lo >= hi) continue;
    const u32 end = hi;
    while (lo < hi) {
      const u32 mid = lo + ((hi - lo) >> 1);
      if (row_blk[mid - q_lo] < (u32)j) lo = mid + 1; else hi = mid;
    }
    if (lo < end && row_blk[lo - q_lo] == (u32)j) present[j] = 1;
  }
}
__global__ void k_shard_dia_add(const unsigned char* __restrict__ present, u32 n, u32* __restrict__ add) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j <= n; j += stride) add[j] = (j < n && !present[j]) ? 1u : 0u;
}
// P_own[0] = 0, P_own[j + 1] = pos[j] + addscan[j]: the A + I column offsets as LinkStream::P (P[x] = pos2[x - 1])
__global__ void k_shard_dia_pos(const u32* __restrict__ pos, const u32* __restrict__ addscan, u32 n, u32* __restrict__ P_own) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j <= n; j += stride) {
    if (j == 0) P_own[0] = 0;
    P_own[j + 1] = pos[j] + addscan[j];
  }
}
// bnd[r] = first A + I position of rank r's block, r = 0..world (bnd[world] = N2)
__global__ void k_shard_dia_bounds(const u32* __restrict__ pos, const u32* __restrict__ addscan, u32 n, u32 N, u32 cnt, int world, u32* __restrict__ bnd) {
  const int r = threadIdx.x;
  if (r > world) return;
  const u64 q = min((u64)N, (u64)r * cnt);
  u32 b;
  if (r == 0) b = 0;
  else if (q >= N) b = N + addscan[n];
  else b = (u32)q + addscan[column_of(pos, n, (u32)q)];
  bnd[r] = b;
}
// the block's real rows at their A + I positions, then its virtual diagonals
__global__ void k_shard_dia_rows(const u32* __restrict__ pos, const u32* __restrict__ addscan, u32 n, const u32* __restrict__ row_blk, u32 q_lo,
                                 size_t cntL, u32 b_lo, u32* __restrict__ row2) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < cntL; p += stride) {
    const u32 q = q_lo + (u32)p;
    row2[q + __ldg(addscan + column_of(pos, n, q)) - b_lo] = row_blk[p];
  }
}
__global__ void k_shard_dia_diag(const u32* __restrict__ P_own, const u32* __restrict__ add, u32 n, u32 b_lo, u32 b_hi, u32* __restrict__ row2) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) {
    if (!add[j]) continue;
    const u32 d = P_own[j + 2] - 1;  // pos2[j + 1] - 1: the end of column j (k_aug_diag)
    if (d >= b_lo && d < b_hi) row2[d - b_lo] = (u32)j;
  }
}

struct DiaLayout {
  DBuf<u32> add, addscan, P_own;
  std::vector<u32> bnd;  // [world + 1] A + I block boundaries
  size_t N2 = 0;
};
// from the combined "diagonal present" flags: addscan, the A + I column offsets and every rank's A + I block
static void dia_layout(const Matrix& A, const unsigned char* present, int world, i64 cnt, DiaLayout& L) {
  const u32 n = (u32)A.n;
  L.add.alloc((size_t)n + 1);
  L.addscan.alloc((size_t)n + 1);
  L.P_own.alloc((size_t)n + 2);
  CPB_LAUNCH(k_shard_dia_add, grid_for((size_t)n + 1), 256, 0, present, n, L.add.get());
  exclusive_scan_u32(L.add.get(), L.addscan.get(), (size_t)n + 1);
  CPB_LAUNCH(k_shard_dia_pos, grid_for((size_t)n + 1), 256, 0, A.pos.get(), L.addscan.get(), n, L.P_own.get());
  DBuf<u32> bnd((size_t)world + 1);
  CPB_LAUNCH(k_shard_dia_bounds, 1, 32, 0, A.pos.get(), L.addscan.get(), n, (u32)A.N, (u32)cnt, world, bnd.get());
  L.bnd.assign((size_t)world + 1, 0u);
  CPB_CUDA(cudaMemcpyAsync(L.bnd.data(), bnd.get(), ((size_t)world + 1) * sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  L.N2 = L.bnd[world];
}
// rank r's rows of A + I (rows of its A block [q_lo, q_lo + cntL) plus the virtual diagonals that fall into its A + I block)
static void dia_block_rows(const Matrix& A, const DiaLayout& L, const u32* P_own, const u32* row_blk, i64 q_lo, size_t cntL, int r, DBuf<u32>& out) {
  const u32 n = (u32)A.n, b_lo = L.bnd[r], b_hi = L.bnd[r + 1];
  out.alloc(std::max<size_t>(b_hi - b_lo, 1));
  if (cntL) CPB_LAUNCH(k_shard_dia_rows, grid_for(cntL), 256, 0, A.pos.get(), L.addscan.get(), n, row_blk, (u32)q_lo, cntL, b_lo, out.get());
  if (n && b_hi > b_lo) CPB_LAUNCH(k_shard_dia_diag, grid_for(n), 256, 0, P_own, L.add.get(), n, b_lo, b_hi, out.get());
}

// link stream of A (dia = nullptr: P = A.pos) or of A + I (P = the layout's offsets, taken over)
static std::unique_ptr<LinkStream> new_link_stream(const Matrix& A, size_t min_entries, DiaLayout* dia) {
  const size_t Ne = dia ? dia->N2 : (size_t)A.N;
  auto ls = std::make_unique<LinkStream>();
  ls->pos_links = true;
  ls->Ne = Ne;
  ls->prev.alloc(std::max<size_t>(Ne, min_entries));
  ls->first_count.alloc(2);
  CPB_CUDA(cudaMemsetAsync(ls->first_count.get(), 0, 2 * sizeof(u32), ctx().stream));
  if (dia) {
    ls->P_own = std::move(dia->P_own);
    ls->P = ls->P_own.get();
  } else {
    ls->P = A.pos.get() - 1;
  }
  fill_colq(*ls, (u32)A.n);
  ls->speculative = false;
  return ls;
}

// the complete link stream of the sharded matrix (dia: of A + I) on every rank
static std::unique_ptr<LinkStream> sharded_link_stream(const ShardedMatrix& S, bool dia) {
  const Matrix& A = S.M;
  const size_t m = (size_t)A.m;
  const u32 n = (u32)A.n;
  const u32* rows = S.row_blk.get();
  size_t cntL = (size_t)(S.q_hi - S.q_lo);
  u32 off = (u32)S.q_lo;
  DiaLayout L;
  DBuf<u32> rows2;
  if (dia) {
    ProfScope pk("shard_dia", (double)n);
    DBuf<unsigned char> present(std::max<size_t>(n, 1));
    present.zero();
    if (n) CPB_LAUNCH(k_shard_diag_present, grid_for(n), 256, 0, A.pos.get(), rows, n, (u32)S.q_lo, (u32)S.q_hi, present.get());
    if (S.world > 1 && n) CPB_NCCL(g_nccl.AllReduce(present.get(), present.get(), n, ncclUint8, ncclMax, g_comm, ctx().stream));
    dia_layout(A, present.get(), S.world, S.cnt, L);  // (synchronises: `present` is free afterwards)
  }
  auto ls = new_link_stream(A, dia ? 0 : (size_t)S.cnt * S.world, dia ? &L : nullptr);
  if (dia) {
    dia_block_rows(A, L, ls->P_own.get(), rows, S.q_lo, cntL, S.rank, rows2);
    rows = rows2.get();
    off = L.bnd[S.rank];
    cntL = L.bnd[S.rank + 1] - L.bnd[S.rank];
  }
  BlockWork w;
  block_local_links(rows, cntL, off, m, ls->prev.get(), w);
  DBuf<u32> carry(std::max<size_t>(m, 1));
  const bool has_in = S.rank > 0 && S.world > 1;
  if (S.world > 2 && std::getenv("CPB_SHARD_CHAIN") == nullptr) {
    // every rank needs the last position of each row in the blocks LEFT of its own.  More than two ranks: one all-gather
    // of the per-block "last position" arrays (world x m x 4 bytes in, m x 4 bytes out per rank) and a local pick of the
    // nearest non-empty entry -- all ranks finish together instead of waiting for a chain of world - 1 hops.
    ProfScope pk("shard_carry", (double)m * 4.0 * S.world);
    DBuf<u32> all(std::max<size_t>(m, 1) * S.world);
    CPB_NCCL(g_nccl.AllGather(w.last_local.get(), all.get(), m, ncclUint32, g_comm, ctx().stream));
    if (has_in) CPB_LAUNCH(k_carry_pick, grid_for(m), 256, 0, all.get(), m, S.rank, carry.get());
    block_heads(w, has_in ? carry.get() : nullptr, off, ls->prev.get(), ls->first_count.get());
    CPB_CUDA(cudaStreamSynchronize(ctx().stream));  // `all` is released at the end of this scope
  } else {
    // two ranks (or CPB_SHARD_CHAIN=1): the "last seen" array travels down the ranks once, m * 4 bytes per hop
    ProfScope pk("shard_carry", (double)m * 4.0);
    if (has_in) CPB_NCCL(g_nccl.Recv(carry.get(), m, ncclUint32, S.rank - 1, g_comm, ctx().stream));
    if (S.rank + 1 < S.world) {
      DBuf<u32> out(std::max<size_t>(m, 1));
      CPB_LAUNCH(k_carry_merge, grid_for(m), 256, 0, w.last_local.get(), has_in ? carry.get() : nullptr, out.get(), m);
      CPB_NCCL(g_nccl.Send(out.get(), m, ncclUint32, S.rank + 1, g_comm, ctx().stream));
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));  // `out` is released at the end of this scope
    }
    block_heads(w, has_in ? carry.get() : nullptr, off, ls->prev.get(), ls->first_count.get());
  }
  if (S.world > 1) {
    ProfScope pk("shard_allgather", (double)(dia ? L.N2 : (size_t)S.cnt * S.world) * 4.0);
    CPB_NCCL(g_nccl.GroupStart());
    if (dia) {
      // the A + I blocks differ in size by their virtual diagonals: one in-place broadcast per rank at its offset
      for (int r = 0; r < S.world; ++r) {
        const size_t len = L.bnd[r + 1] - L.bnd[r];
        u32* const p = ls->prev.get() + L.bnd[r];
        if (len) CPB_NCCL(g_nccl.Broadcast(p, p, len, ncclUint32, r, g_comm, ctx().stream));
      }
    } else {
      CPB_NCCL(g_nccl.AllGather(ls->prev.get() + (size_t)S.rank * S.cnt, ls->prev.get(), (size_t)S.cnt, ncclUint32, g_comm, ctx().stream));
    }
    CPB_NCCL(g_nccl.AllReduce(ls->first_count.get(), ls->first_count.get(), 1, ncclUint32, ncclSum, g_comm, ctx().stream));
    CPB_NCCL(g_nccl.GroupEnd());
  }
  return ls;
}

// The same construction with the ranks played one after the other on this GPU (tests: the block kernels and the carry rule
// without NCCL).  A holds the complete pattern; dia: the link stream of A + I with the blocks of sharded_link_stream.
std::unique_ptr<LinkStream> emulated_sharded_link_stream(const Matrix& A, int world, bool dia) {
  const size_t m = (size_t)A.m;
  const u32 n = (u32)A.n;
  i64 cnt = 0;
  shard_range(A.N, 0, world, &cnt, nullptr, nullptr);
  DiaLayout L;
  if (dia) {
    DBuf<unsigned char> present(std::max<size_t>(n, 1));
    present.zero();
    for (int r = 0; r < world && n; ++r) {
      i64 lo = 0, hi = 0;
      shard_range(A.N, r, world, nullptr, &lo, &hi);
      if (hi > lo) CPB_LAUNCH(k_shard_diag_present, grid_for(n), 256, 0, A.pos.get(), A.row.get() + lo, n, (u32)lo, (u32)hi, present.get());
    }
    dia_layout(A, present.get(), world, cnt, L);
  }
  auto ls = new_link_stream(A, dia ? 0 : (size_t)cnt * world, dia ? &L : nullptr);
  // rank r's rows and their first (A or A + I) position
  auto block = [&](int r, DBuf<u32>& tmp, const u32*& rows, size_t& len, u32& off) {
    i64 lo = 0, hi = 0;
    shard_range(A.N, r, world, nullptr, &lo, &hi);
    rows = A.row.get() + lo;
    len = (size_t)(hi - lo);
    off = (u32)lo;
    if (dia) {
      dia_block_rows(A, L, ls->P_own.get(), rows, lo, len, r, tmp);
      rows = tmp.get();
      off = L.bnd[r];
      len = L.bnd[r + 1] - L.bnd[r];
    }
  };
  DBuf<u32> carry(std::max<size_t>(m, 1)), next(std::max<size_t>(m, 1));
  const bool pick = world > 2 && std::getenv("CPB_SHARD_CHAIN") == nullptr;  // the same two carry forms as the real ranks
  if (pick) {
    // pass 1: every block's local links and last positions; pass 2: heads from the nearest non-empty entry below
    DBuf<u32> all(std::max<size_t>(m, 1) * world);
    std::vector<BlockWork> ws(world);
    std::vector<u32> offs(world);
    for (int r = 0; r < world; ++r) {
      DBuf<u32> tmp;
      const u32* rows = nullptr;
      size_t len = 0;
      block(r, tmp, rows, len, offs[r]);
      block_local_links(rows, len, offs[r], m, ls->prev.get(), ws[r]);
      if (m) CPB_CUDA(cudaMemcpyAsync(all.get() + (size_t)r * m, ws[r].last_local.get(), m * sizeof(u32), cudaMemcpyDeviceToDevice, ctx().stream));
    }
    for (int r = 0; r < world; ++r) {
      if (r > 0) CPB_LAUNCH(k_carry_pick, grid_for(m), 256, 0, all.get(), m, r, carry.get());
      block_heads(ws[r], r > 0 ? carry.get() : nullptr, offs[r], ls->prev.get(), ls->first_count.get());
    }
    CPB_CUDA(cudaStreamSynchronize(ctx().stream));  // the blocks' buffers are released here
    return ls;
  }
  for (int r = 0; r < world; ++r) {
    DBuf<u32> tmp;
    const u32* rows = nullptr;
    size_t len = 0;
    u32 off = 0;
    block(r, tmp, rows, len, off);
    BlockWork w;
    block_local_links(rows, len, off, m, ls->prev.get(), w);
    block_heads(w, r > 0 ? carry.get() : nullptr, off, ls->prev.get(), ls->first_count.get());
    CPB_LAUNCH(k_carry_merge, grid_for(m), 256, 0, w.last_local.get(), r > 0 ? carry.get() : nullptr, next.get(), m);
    std::swap(carry, next);
    CPB_CUDA(cudaStreamSynchronize(ctx().stream));  // the block's buffers are released here
  }
  return ls;
}

ShardedMatrix* sharded_create(i64 m, i64 n, i64 nnz, const i64* h_colptr, const i64* h_rowval, bool rows_are_block,
                              void (*upload)(const i64*, size_t, u32*, i64, i64, u32*)) {
  CPB_REQUIRE(g_comm != nullptr || g_world == 1, "call cpb_comm_init first");
  CPB_REQUIRE(m >= 0 && n >= 0 && nnz >= 0, "negative dimension");
  CPB_REQUIRE(nnz + n + 1 < ((i64)1 << 31) && m < ((i64)1 << 31) - 2 && n < ((i64)1 << 31) - 2, "matrix too large for the 32-bit device index");
  auto S = std::make_unique<ShardedMatrix>();
  S->rank = g_rank;
  S->world = g_world;
  S->M.m = m; S->M.n = n; S->M.N = nnz;
  shard_range(nnz, g_rank, g_world, &S->cnt, &S->q_lo, &S->q_hi);
  const size_t cntL = (size_t)(S->q_hi - S->q_lo);
  // the column offsets are needed whole on every rank: each rank uploads one slice, one in-place all-gather completes them
  // (the ranks share the host's memory bandwidth -- n + 1 Int64 values read once instead of `world` times)
  i64 ccnt = 0, clo = 0, chi = 0;
  shard_range(n + 1, g_rank, g_world, &ccnt, &clo, &chi);
  S->M.pos.alloc(std::max<size_t>((size_t)n + 1, (size_t)ccnt * g_world));
  S->row_blk.alloc(std::max<size_t>(cntL, 1));
  DBuf<u32> flags(1);
  flags.zero();
  if (g_world > 1 && g_comm) {
    if (chi > clo) upload(h_colptr + clo, (size_t)(chi - clo), S->M.pos.get() + clo, 1, nnz + 1, flags.get());
    CPB_NCCL(g_nccl.AllGather(S->M.pos.get() + (size_t)g_rank * ccnt, S->M.pos.get(), (size_t)ccnt, ncclUint32, g_comm, ctx().stream));
  } else {
    upload(h_colptr, (size_t)n + 1, S->M.pos.get(), 1, nnz + 1, flags.get());
  }
  if (cntL) upload(rows_are_block ? h_rowval : h_rowval + S->q_lo, cntL, S->row_blk.get(), 1, m, flags.get());
  check_monotone(S->M.pos.get(), (size_t)n + 1, flags.get());
  if (g_world > 1 && g_comm) CPB_NCCL(g_nccl.AllReduce(flags.get(), flags.get(), 1, ncclUint32, ncclMax, g_comm, ctx().stream));  // every rank fails together
  u32 hf = 0;
  CPB_CUDA(cudaMemcpyAsync(&hf, flags.get(), sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  CPB_REQUIRE((hf & 1u) == 0, "colptr/rowval entry out of range (expected 1-based indices)");
  CPB_REQUIRE((hf & 2u) == 0, "colptr is not non-decreasing");
  CPB_REQUIRE(h_colptr[0] == 1 && h_colptr[n] == nnz + 1, "colptr[1] must be 1 and colptr[n+1] must be nnz+1");
  return S.release();
}

void sharded_destroy(ShardedMatrix* S) { delete S; }

void sharded_dims(const ShardedMatrix& S, i64* m, i64* n, i64* nnz, i64* q_lo, i64* q_hi) {
  if (m) *m = S.M.m;
  if (n) *n = S.M.n;
  if (nnz) *nnz = S.M.N;
  if (q_lo) *q_lo = S.q_lo;
  if (q_hi) *q_hi = S.q_hi;
}

void bisect_node_buffers(BisectRun& run, int** res, double** c, int** spl, int* P);  // bisect.cu
bool bisect_is_done(BisectRun& run);

static bool sharded_model(const cpb_model* mdl) { return mdl && (mdl->kind == CPB_MODEL_CONNECTIVITY || mdl->kind == CPB_MODEL_MONOSYM); }

void solve_sharded(ShardedMatrix& S, const cpb_model* mdl, int method, double eps, i64 K, int64_t* h_spl_out) {
  CPB_REQUIRE(method == CPB_SPLIT_BISECT_COST || method == CPB_SPLIT_LAZY_BISECT_COST, "sharded solves: BisectCost / LazyBisectCost splitters");
  CPB_REQUIRE(sharded_model(mdl), "sharded solves: AffineConnectivityModel or AffineMonotonizedSymmetricConnectivityModel (the streaming link forms)");
  CPB_REQUIRE(S.world == g_world && S.rank == g_rank, "the sharded matrix was created under another communicator");
  const double t0 = now_ms();
  auto f = oracle_create(S.M, mdl, nullptr, 0);  // (the monotonized symmetric model checks that A is square, on every rank alike)
  const bool dia = mdl->kind == CPB_MODEL_MONOSYM;
  f->ls = sharded_link_stream(S, dia);
  const double t1 = now_ms();
  const int cap = std::min(probe_cluster_capacity(true), 15);
  const int per = std::max(1, std::min(cap, 255 / S.world));
  const int nodes = per * S.world;
  BisectRunPtr run = bisect_begin(*f, method == CPB_SPLIT_LAZY_BISECT_COST, eps, K, nodes);
  int rounds = 0;
  double coll_bytes = 0;
  {
    ProfScope prof("probe");
    int* res = nullptr;
    double* c = nullptr;
    int* spl = nullptr;
    int P = 0;
    bisect_node_buffers(*run, &res, &c, &spl, &P);
    CPB_REQUIRE(P == nodes, "speculation tree size mismatch");
    bool done = false;
    for (int guard = 0; guard < 4096; ++guard) {
      if (bisect_is_done(*run)) { done = true; break; }
      bisect_probe(*run, S.rank * per, (S.rank + 1) * per);
      if (S.world > 1) {
        ProfScope pk("shard_threshold_allgather", (double)nodes * (12.0 + 4.0 * (K + 2)));
        CPB_NCCL(g_nccl.GroupStart());
        CPB_NCCL(g_nccl.AllGather(res + S.rank * per, res, (size_t)per, ncclInt32, g_comm, ctx().stream));
        CPB_NCCL(g_nccl.AllGather(c + S.rank * per, c, (size_t)per, ncclFloat64, g_comm, ctx().stream));
        CPB_NCCL(g_nccl.AllGather(spl + (size_t)S.rank * per * (K + 2), spl, (size_t)per * (K + 2), ncclInt32, g_comm, ctx().stream));
        CPB_NCCL(g_nccl.GroupEnd());
        coll_bytes += (double)nodes * (12.0 + 4.0 * (K + 2));
      }
      ++rounds;
      if (bisect_advance(*run, true)) { done = true; break; }
    }
    CPB_REQUIRE(done, "bisection did not terminate (eps too small for Float64?)");
  }
  bisect_finish(*run, h_spl_out);
  const double t2 = now_ms();
  g_shard_stats[0] = S.world;
  g_shard_stats[1] = t1 - t0;                      // link construction incl. carry + all-gather, host clock (asynchronous part excluded)
  g_shard_stats[2] = t2 - t1;                      // bisection (includes waiting for the construction queued before it)
  g_shard_stats[3] = rounds;
  g_shard_stats[4] = (double)(dia ? f->ls->Ne : (size_t)S.cnt * S.world) * 4.0;  // link gather bytes (whole array; A + I for dia)
  g_shard_stats[5] = (double)S.M.m * 4.0;          // carry bytes per hop
  g_shard_stats[6] = coll_bytes;                   // threshold all-gather bytes
  g_shard_stats[7] = nodes;
}

// single-GPU stand-in for `world` ranks: emulated block construction, every threshold slot probed here (tests)
void solve_sharded_emulated(Matrix& A, const cpb_model* mdl, int method, double eps, i64 K, int world, int64_t* h_spl_out) {
  CPB_REQUIRE(method == CPB_SPLIT_BISECT_COST || method == CPB_SPLIT_LAZY_BISECT_COST, "sharded solves: BisectCost / LazyBisectCost splitters");
  CPB_REQUIRE(sharded_model(mdl), "sharded solves: AffineConnectivityModel or AffineMonotonizedSymmetricConnectivityModel (the streaming link forms)");
  CPB_REQUIRE(world >= 1 && world <= 16, "1..16 emulated ranks");
  auto f = oracle_create(A, mdl, nullptr, 0);
  f->ls = emulated_sharded_link_stream(A, world, mdl->kind == CPB_MODEL_MONOSYM);
  const int cap = std::min(probe_cluster_capacity(true), 15);
  const int per = std::max(1, std::min(cap, 255 / world));
  BisectRunPtr run = bisect_begin(*f, method == CPB_SPLIT_LAZY_BISECT_COST, eps, K, per * world);
  bool done = false;
  for (int guard = 0; guard < 4096 && !done; ++guard) {
    if (bisect_is_done(*run)) break;
    for (int r = 0; r < world; ++r) bisect_probe(*run, r * per, (r + 1) * per);
    done = bisect_advance(*run, true);
  }
  bisect_finish(*run, h_spl_out);
}

// ---- adjointpattern of a sharded matrix ---------------------------------------------------------------------------------
// Aᵀ has the same nnz, so the same shard_range blocks.  Rank r sorts its block by row (stable: columns ascend inside a row);
// the per-block row histograms (m x 4 bytes each) are all-gathered, which gives every rank colptrᵀ (their sum) and
// below[i] (the sum over the lower ranks).  The Aᵀ position of the block's k-th entry of row i is
// colptrᵀ[i] + below[i] + k.  Those positions increase along the sorted block, so each destination rank receives one
// contiguous slice: (column << 32 | position) pairs, 8 bytes per nonzero, grouped ncclSend / ncclRecv, scattered there.
__global__ void k_tr_hist(const u32* __restrict__ rows, size_t cnt, u32* __restrict__ hist) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < cnt; p += stride) atomicAdd(&hist[rows[p]], 1u);
}
// tot[i] = entries of row i over all blocks, below[i] = over the blocks of the ranks below `rank`
__global__ void k_tr_combine(const u32* __restrict__ all, size_t m, int world, int rank, u32* __restrict__ tot, u32* __restrict__ below) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) {
    u32 t = 0, b = 0;
    for (int r = 0; r < world; ++r) {
      if (r == rank) b = t;
      t += all[(size_t)r * m + i];
    }
    tot[i] = t;
    below[i] = b;
  }
}
// the sorted block (packed pairs of the one-sweep sort, or keys / values) -> (column << 32 | Aᵀ position) in sorted order
__global__ void k_tr_pairs(const u64* __restrict__ sorted, const u32* __restrict__ sk, const u32* __restrict__ sq, size_t cntL, u32 q_lo,
                           const u32* __restrict__ pos, u32 n, const u32* __restrict__ colptrT, const u32* __restrict__ below,
                           const u32* __restrict__ lstart, u64* __restrict__ out) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < cntL; p += stride) {
    u32 i, lp;
    if (sorted) {
      const u64 v = sorted[p];
      i = (u32)(v >> 32);
      lp = (u32)v;
    } else {
      i = sk[p];
      lp = sq[p];
    }
    const u32 dst = colptrT[i] + below[i] + ((u32)p - lstart[i]);
    out[p] = ((u64)column_of(pos, n, q_lo + lp) << 32) | dst;
  }
}
// off[d] = first pair bound for rank d's block or a later one (d = 0..world); counts[d] = off[d + 1] - off[d]
__global__ void k_tr_slices(const u64* __restrict__ pairs, size_t cntL, u64 cnt, u64 N, int world, u32* __restrict__ off, u32* __restrict__ counts) {
  __shared__ u32 s[33];
  const int d = threadIdx.x;
  if (d <= world) {
    const u64 t = min(N, (u64)d * cnt);
    size_t lo = 0, hi = cntL;
    while (lo < hi) {
      const size_t mid = lo + ((hi - lo) >> 1);
      if ((u64)(u32)pairs[mid] < t) lo = mid + 1; else hi = mid;
    }
    s[d] = (u32)lo;
    off[d] = (u32)lo;
  }
  __syncthreads();
  if (d < world && counts) counts[d] = s[d + 1] - s[d];
}
__global__ void k_tr_scatter(const u64* __restrict__ pairs, size_t cnt, u32 q_lo, u32* __restrict__ row_blk) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < cnt; p += stride) {
    const u64 v = pairs[p];
    row_blk[(u32)v - q_lo] = (u32)(v >> 32);
  }
}

struct TrBlock {
  DBuf<u32> k0, v0, k1, v1;
  DBuf<u64> a, b;
  const u64* sorted = nullptr;
  const u32 *sk = nullptr, *sq = nullptr;
};
// stable sort of a block by row: the one-sweep passes block_local_links runs, or the tile-histogram sort
static void tr_sort(const u32* rows, size_t cntL, size_t m, TrBlock& t) {
  if (!cntL) return;
  const char* os_env = std::getenv("CPB_ONESWEEP");
  if (onesweep_supported(cntL) && !(os_env && os_env[0] == '0')) {
    t.a.alloc(cntL);
    t.b.alloc(cntL);
    t.sorted = onesweep_sort_iota(rows, cntL, bits_for(m ? m - 1 : 0), t.a.get(), t.b.get());
    return;
  }
  t.k0.alloc(cntL); t.v0.alloc(cntL); t.k1.alloc(cntL); t.v1.alloc(cntL);
  const int which = radix_sort_pairs_iota(rows, t.k0.get(), t.v0.get(), t.k1.get(), t.v1.get(), cntL, bits_for(m ? m - 1 : 0));
  t.sk = which ? t.k1.get() : t.k0.get();
  t.sq = which ? t.v1.get() : t.v0.get();
}
// colptrᵀ (m + 1, 0-based) and the routed pairs of rank `rank`'s sorted block, from every rank's row histogram (all: world x m)
static void tr_pairs(const Matrix& A, const u32* all, int world, int rank, const TrBlock& t, size_t cntL, u32 q_lo, u32* colptrT, DBuf<u64>& pairs) {
  const size_t m = (size_t)A.m;
  DBuf<u32> tot(m + 1), below(std::max<size_t>(m, 1)), lstart(std::max<size_t>(m, 1));
  tot.zero();
  if (m) {
    CPB_LAUNCH(k_tr_combine, grid_for(m), 256, 0, all, m, world, rank, tot.get(), below.get());
    exclusive_scan_u32(all + (size_t)rank * m, lstart.get(), m);
  }
  exclusive_scan_u32(tot.get(), colptrT, m + 1);
  pairs.alloc(std::max<size_t>(cntL, 1));
  if (cntL) CPB_LAUNCH(k_tr_pairs, grid_for(cntL), 256, 0, t.sorted, t.sk, t.sq, cntL, q_lo, A.pos.get(), (u32)A.n, colptrT, below.get(), lstart.get(), pairs.get());
}

ShardedMatrix* sharded_adjointpattern(const ShardedMatrix& S) {
  CPB_REQUIRE(S.world == g_world && S.rank == g_rank, "the sharded matrix was created under another communicator");
  const Matrix& A = S.M;
  const size_t m = (size_t)A.m, cntL = (size_t)(S.q_hi - S.q_lo);
  const int world = S.world, rank = S.rank;
  ProfScope prof("shard_adjointpattern", (double)cntL * 16.0 + (double)m * 4.0 * world);
  auto T = std::make_unique<ShardedMatrix>();
  T->rank = rank;
  T->world = world;
  T->M.m = A.n; T->M.n = A.m; T->M.N = A.N;
  T->cnt = S.cnt; T->q_lo = S.q_lo; T->q_hi = S.q_hi;
  T->M.pos.alloc(m + 1);
  T->row_blk.alloc(std::max<size_t>(cntL, 1));
  DBuf<u32> all(std::max<size_t>(m, 1) * world);
  all.zero();
  u32* const mine = all.get() + (size_t)rank * m;
  if (cntL) CPB_LAUNCH(k_tr_hist, grid_for(cntL), 256, 0, S.row_blk.get(), cntL, mine);
  if (world > 1 && m) CPB_NCCL(g_nccl.AllGather(mine, all.get(), m, ncclUint32, g_comm, ctx().stream));
  TrBlock t;
  tr_sort(S.row_blk.get(), cntL, m, t);
  DBuf<u64> pairs;
  tr_pairs(A, all.get(), world, rank, t, cntL, (u32)S.q_lo, T->M.pos.get(), pairs);
  if (world == 1) {
    if (cntL) CPB_LAUNCH(k_tr_scatter, grid_for(cntL), 256, 0, pairs.get(), cntL, 0u, T->row_blk.get());
    CPB_CUDA(cudaStreamSynchronize(ctx().stream));
    return T.release();
  }
  // world x world pair counts: row s = what rank s sends to every rank
  DBuf<u32> off((size_t)world + 1), counts((size_t)world * world);
  CPB_LAUNCH(k_tr_slices, 1, 32, 0, pairs.get(), cntL, (u64)S.cnt, (u64)A.N, world, off.get(), counts.get() + (size_t)rank * world);
  CPB_NCCL(g_nccl.AllGather(counts.get() + (size_t)rank * world, counts.get(), (size_t)world, ncclUint32, g_comm, ctx().stream));
  std::vector<u32> h_off((size_t)world + 1), h_cnt((size_t)world * world);
  CPB_CUDA(cudaMemcpyAsync(h_off.data(), off.get(), h_off.size() * sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaMemcpyAsync(h_cnt.data(), counts.get(), h_cnt.size() * sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  std::vector<size_t> recv_off((size_t)world + 1, 0);
  for (int s = 0; s < world; ++s) recv_off[s + 1] = recv_off[s] + h_cnt[(size_t)s * world + rank];
  CPB_REQUIRE(recv_off[world] == cntL, "sharded adjointpattern: the routed slices do not cover this rank's block");
  DBuf<u64> recv(std::max<size_t>(cntL, 1));
  {
    ProfScope pk("shard_transpose_exchange", (double)cntL * 8.0);
    CPB_NCCL(g_nccl.GroupStart());
    for (int d = 0; d < world; ++d) {
      const size_t c = h_cnt[(size_t)rank * world + d];
      if (d != rank && c) CPB_NCCL(g_nccl.Send(pairs.get() + h_off[d], c, ncclUint64, d, g_comm, ctx().stream));
    }
    for (int s = 0; s < world; ++s) {
      const size_t c = h_cnt[(size_t)s * world + rank];
      if (s != rank && c) CPB_NCCL(g_nccl.Recv(recv.get() + recv_off[s], c, ncclUint64, s, g_comm, ctx().stream));
    }
    CPB_NCCL(g_nccl.GroupEnd());
  }
  const size_t self = h_cnt[(size_t)rank * world + rank];
  if (self)
    CPB_CUDA(cudaMemcpyAsync(recv.get() + recv_off[rank], pairs.get() + h_off[rank], self * sizeof(u64), cudaMemcpyDeviceToDevice, ctx().stream));
  if (cntL) CPB_LAUNCH(k_tr_scatter, grid_for(cntL), 256, 0, recv.get(), cntL, (u32)S.q_lo, T->row_blk.get());
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));  // the exchange buffers are released at the end of this scope
  g_shard_stats[8] = (double)(cntL - self) * 8.0;  // transpose pairs received from other ranks (bytes, this rank)
  g_shard_stats[9] = (double)m * 4.0 * world;      // histogram all-gather bytes
  return T.release();
}

// The same with the ranks played one after the other on this GPU; assembles the whole Aᵀ (tests)
std::unique_ptr<Matrix> adjoint_pattern_sharded_emulated(const Matrix& A, int world) {
  CPB_REQUIRE(world >= 1 && world <= 16, "1..16 emulated ranks");
  const size_t m = (size_t)A.m, N = (size_t)A.N;
  i64 cnt = 0;
  shard_range(A.N, 0, world, &cnt, nullptr, nullptr);
  auto B = std::make_unique<Matrix>();
  B->m = A.n; B->n = A.m; B->N = A.N;
  B->pos.alloc(m + 1);
  B->row.alloc(N);
  DBuf<u32> all(std::max<size_t>(m, 1) * world);
  all.zero();
  for (int r = 0; r < world; ++r) {
    i64 lo = 0, hi = 0;
    shard_range(A.N, r, world, nullptr, &lo, &hi);
    if (hi > lo) CPB_LAUNCH(k_tr_hist, grid_for((size_t)(hi - lo)), 256, 0, A.row.get() + lo, (size_t)(hi - lo), all.get() + (size_t)r * m);
  }
  DBuf<u32> colptrT(m + 1), off((size_t)world + 1);
  for (int r = 0; r < world; ++r) {
    i64 lo = 0, hi = 0;
    shard_range(A.N, r, world, nullptr, &lo, &hi);
    const size_t cntL = (size_t)(hi - lo);
    TrBlock t;
    tr_sort(A.row.get() + lo, cntL, m, t);
    DBuf<u64> pairs;
    tr_pairs(A, all.get(), world, r, t, cntL, (u32)lo, r == 0 ? B->pos.get() : colptrT.get(), pairs);
    // the slices as the destination ranks would receive them
    CPB_LAUNCH(k_tr_slices, 1, 32, 0, pairs.get(), cntL, (u64)cnt, (u64)N, world, off.get(), (u32*)nullptr);
    std::vector<u32> h_off((size_t)world + 1);
    CPB_CUDA(cudaMemcpyAsync(h_off.data(), off.get(), h_off.size() * sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
    CPB_CUDA(cudaStreamSynchronize(ctx().stream));
    for (int d = 0; d < world; ++d) {
      i64 dlo = 0;
      shard_range(A.N, d, world, nullptr, &dlo, nullptr);
      const size_t c = h_off[d + 1] - h_off[d];
      if (c) CPB_LAUNCH(k_tr_scatter, grid_for(c), 256, 0, pairs.get() + h_off[d], c, (u32)dlo, B->row.get() + dlo);
    }
    CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  }
  return B;
}

// colptr (n + 1) and this rank's block of rowval, both 1-based
void sharded_get(const ShardedMatrix& S, i64* h_colptr, i64* h_rowval_blk) {
  const size_t n = (size_t)S.M.n, cntL = (size_t)(S.q_hi - S.q_lo);
  DBuf<i64> dc(n + 1), dr(std::max<size_t>(cntL, 1));
  if (h_colptr) {
    widen_plus(S.M.pos.get(), dc.get(), n + 1, 1);
    CPB_CUDA(cudaMemcpyAsync(h_colptr, dc.get(), (n + 1) * sizeof(i64), cudaMemcpyDeviceToHost, ctx().stream));
  }
  if (h_rowval_blk && cntL) {
    widen_plus(S.row_blk.get(), dr.get(), cntL, 1);
    CPB_CUDA(cudaMemcpyAsync(h_rowval_blk, dr.get(), cntL * sizeof(i64), cudaMemcpyDeviceToHost, ctx().stream));
  }
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
}

void sharded_stats(double out[16]) {
  for (int t = 0; t < 16; ++t) out[t] = g_shard_stats[t];
}

}  // namespace cpb
