// capi.cu -- the C ABI of libchainb200.so (include/chainb200.h): argument checking, handle
// ownership, error translation.  Nothing throws across this boundary.
#include <algorithm>
#include <chrono>
#include <mutex>
#include <thread>
#include "engine.cuh"
#include "primitives.cuh"

using namespace cpb;

struct cpb_matrix { Matrix M; };
struct cpb_oracle { std::unique_ptr<Oracle> O; };
struct cpb_prefix { std::unique_ptr<PrefixMatrix> P; };

namespace cpb {

static Context g_ctx;
static std::mutex g_mu;
static thread_local std::string g_err;

struct PendingProf {
  std::string name;
  cudaEvent_t e0, e1;
  double bytes;
  i64 launches;
};
static std::vector<PendingProf> g_pending;

Context& ctx() { return g_ctx; }

static void init_context(int device) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0)
    throw Error(CPB_ERR_CUDA, std::string("no usable CUDA device (libchainb200 has no CPU fallback): ") + cudaGetErrorString(e));
  if (device < 0 || device >= count) throw Error(CPB_ERR_ARG, "device index out of range");
  CPB_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  CPB_CUDA(cudaGetDeviceProperties(&prop, device));
  if (g_ctx.stream && g_ctx.device != device) {
    // switching devices: the cached large blocks belong to the old device -- hand them back before anything can reuse them
    // (handles created on the old device stay valid only on it: chainb200.h, "Lifetimes")
    cudaSetDevice(g_ctx.device);
    cudaStreamSynchronize(g_ctx.stream);
    big_trim();
    cudaStreamDestroy(g_ctx.stream);
    g_ctx.stream = nullptr;
    CPB_CUDA(cudaSetDevice(device));
  }
  g_ctx.device = device;
  g_ctx.sm_count = prop.multiProcessorCount;
  if (!g_ctx.stream) CPB_CUDA(cudaStreamCreateWithFlags(&g_ctx.stream, cudaStreamNonBlocking));
  cudaMemPool_t pool;
  CPB_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
  unsigned long long thr = ~0ull;  // keep freed blocks cached in the pool
  CPB_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
  g_ctx.ready = true;
}

// ---- CPB_TRACE ------------------------------------------------------------------------------------------------------
static std::vector<std::pair<const char*, double>> g_trace;
static int trace_on() {
  static const int on = std::getenv("CPB_TRACE") ? std::atoi(std::getenv("CPB_TRACE")) : 0;
  return on;
}
void trace_mark(const char* label) {
  if (!trace_on()) return;
  if (g_ctx.stream) cudaStreamSynchronize(g_ctx.stream);
  g_trace.push_back({label, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count()});
}
void trace_flush(const char* what) {
  if (!trace_on() || g_trace.empty()) return;
  std::string line = std::string("[cpb trace] ") + what + ":";
  for (size_t i = 1; i < g_trace.size(); ++i) {
    char buf[96];
    std::snprintf(buf, sizeof(buf), " %s=%.2f", g_trace[i].first, g_trace[i].second - g_trace[i - 1].second);
    line += buf;
  }
  char buf[64];
  std::snprintf(buf, sizeof(buf), " | total=%.2f ms", g_trace.back().second - g_trace.front().second);
  std::fprintf(stderr, "%s%s\n", line.c_str(), buf);
  g_trace.clear();
}

// ---- free list of large device blocks (see common.cuh) --------------------------------------------------------------
static std::multimap<size_t, void*> g_big_free;
static size_t g_big_cached = 0;
void big_trim() {
  if (g_big_free.empty()) return;
  cudaStreamSynchronize(g_ctx.stream);
  for (auto& kv : g_big_free) cudaFree(kv.second);
  g_big_free.clear();
  g_big_cached = 0;
}
void* big_alloc(size_t bytes) {
  auto it = g_big_free.find(bytes);
  if (it != g_big_free.end()) {
    void* p = it->second;
    g_big_free.erase(it);
    g_big_cached -= bytes;
    return p;
  }
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) {  // give the cached blocks (and the driver pool's) back and try once more
    cudaGetLastError();
    big_trim();
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, g_ctx.device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
    e = cudaMalloc(&p, bytes);
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    throw Error(CPB_ERR_CUDA, std::string("out of device memory (") + std::to_string(bytes >> 20) + " MiB requested): " + cudaGetErrorString(e));
  }
  return p;
}
void big_free(void* p, size_t bytes) {
  // everything is returned to the driver once the cache holds more than a quarter of the device
  static size_t limit = 0;
  if (limit == 0) {
    size_t free_b = 0, total_b = 0;
    limit = (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && total_b > 0) ? total_b / 4 : ((size_t)16 << 30);
  }
  if (g_big_cached + bytes > limit) big_trim();
  g_big_free.emplace(bytes, p);
  g_big_cached += bytes;
}

void ensure_context() {
  if (!g_ctx.ready) init_context(0);
  else CPB_CUDA(cudaSetDevice(g_ctx.device));
}

ProfScope::ProfScope(const char* nm, double algorithmic_bytes) : name(nm), bytes(algorithmic_bytes), launches0(ctx().launches), on(ctx().profiling) {
  if (on) {
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaEventRecord(e0, ctx().stream);
  }
}
ProfScope::~ProfScope() {
  if (on) {
    cudaEventRecord(e1, ctx().stream);
    g_pending.push_back({name, e0, e1, bytes, ctx().launches - launches0});
  }
}

static void resolve_pending() {
  if (g_pending.empty()) return;
  cudaStreamSynchronize(g_ctx.stream);
  for (auto& p : g_pending) {
    float ms = 0;
    cudaEventElapsedTime(&ms, p.e0, p.e1);
    ProfEntry& e = g_ctx.prof_entry(p.name);
    e.ms += ms;
    e.launches += p.launches;
    e.bytes += p.bytes;
    cudaEventDestroy(p.e0);
    cudaEventDestroy(p.e1);
  }
  g_pending.clear();
}

}  // namespace cpb

#define CPB_API_BEGIN                         \
  std::lock_guard<std::mutex> _lk(cpb::g_mu); \
  try {
#define CPB_API_END                      \
  }                                      \
  catch (const cpb::Error& e) {          \
    cpb::g_err = e.what();               \
    return e.code;                       \
  }                                      \
  catch (const std::exception& e) {      \
    cpb::g_err = e.what();               \
    return CPB_ERR_ARG;                  \
  }                                      \
  catch (...) {                          \
    cpb::g_err = "unknown error";        \
    return CPB_ERR_ARG;                  \
  }                                      \
  return CPB_OK;

extern "C" {

const char* cpb_last_error(void) { return cpb::g_err.c_str(); }
int cpb_version(void) { return 101; }

int cpb_init(int device) {
  CPB_API_BEGIN
  init_context(device);
  CPB_API_END
}

int cpb_device_count(void) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess) return 0;
  return count;
}

int cpb_trim_memory(void) {
  CPB_API_BEGIN
  ensure_context();
  big_trim();
  cudaMemPool_t pool;
  CPB_CUDA(cudaDeviceGetDefaultMemPool(&pool, ctx().device));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  CPB_CUDA(cudaMemPoolTrimTo(pool, 0));
  CPB_API_END
}

int cpb_synchronize(void) {
  CPB_API_BEGIN
  ensure_context();
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  CPB_API_END
}

// Host -> device copy of a caller's array.  Pinned (registered) memory goes straight to cudaMemcpyAsync.
// Pageable memory -- what a Julia Array is -- would be staged by the driver through one internal buffer by
// one thread (~10 GB/s measured); instead a pool of host threads (hostpack.cpp) copies chunks into pinned staging
// buffers while the previous chunks are in flight over PCIe.  Int64 index arrays are NARROWED while they are staged
// (upload_index_array below): half the PCIe bytes.
static constexpr size_t H2D_CHUNK = (size_t)32 << 20;
static constexpr size_t PACK_CHUNK_ELEMS = (size_t)2 << 20;  // 8 MB staged / 16 MB of Int64 source per chunk
static constexpr int H2D_BUFS = 4;
static void* g_stage[H2D_BUFS] = {nullptr, nullptr, nullptr, nullptr};
static cudaEvent_t g_stage_ev[H2D_BUFS] = {nullptr, nullptr, nullptr, nullptr};
static bool g_stage_busy[H2D_BUFS] = {false, false, false, false};
static int g_stage_next = 0;

extern "C++" {
namespace cpb {
void host_copy(void* dst, const void* src, size_t bytes);            // hostpack.cpp
uint64_t host_pack(uint32_t* dst, const int64_t* src, size_t n);     // hostpack.cpp
}
}

static bool host_pinned(const void* p) {
  cudaPointerAttributes attr{};
  const bool pinned = cudaPointerGetAttributes(&attr, p) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();  // unregistered memory may set a sticky-free error on old drivers
  return pinned;
}
static bool staging_disabled() {
  static const bool disabled = std::getenv("CPB_NO_STAGED_H2D") != nullptr;
  return disabled;
}
// next staging buffer, free to be overwritten by the host
static int stage_acquire() {
  for (int b = 0; b < H2D_BUFS; ++b)
    if (!g_stage[b]) {
      CPB_CUDA(cudaHostAlloc(&g_stage[b], H2D_CHUNK, cudaHostAllocDefault));
      CPB_CUDA(cudaEventCreateWithFlags(&g_stage_ev[b], cudaEventDisableTiming));
    }
  const int b = g_stage_next;
  g_stage_next = (g_stage_next + 1) % H2D_BUFS;
  if (g_stage_busy[b]) CPB_CUDA(cudaEventSynchronize(g_stage_ev[b]));  // the copy that last used this buffer (maybe in an earlier call) has finished
  return b;
}
static void stage_release(int b) {
  CPB_CUDA(cudaEventRecord(g_stage_ev[b], ctx().stream));
  g_stage_busy[b] = true;
}

static void h2d_copy(void* d_dst, const void* h_src, size_t bytes) {
  if (bytes == 0) return;
  if (host_pinned(h_src) || bytes < 2 * H2D_CHUNK || staging_disabled()) {
    CPB_CUDA(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx().stream));
    return;
  }
  for (size_t off = 0; off < bytes; off += H2D_CHUNK) {
    const int b = stage_acquire();
    const size_t sz = std::min(H2D_CHUNK, bytes - off);
    host_copy(g_stage[b], (const char*)h_src + off, sz);
    CPB_CUDA(cudaMemcpyAsync((char*)d_dst + off, g_stage[b], sz, cudaMemcpyHostToDevice, ctx().stream));
    stage_release(b);
  }
}

// 1-based Int64 host index array -> 0-based u32 device array, range-checked ([lo, hi], flags |= 1 on the device).
// The source is narrowed to 32 bits by the host pool while it is staged, the decrement + check runs per chunk on the
// device behind its copy; short arrays go over the bus as they are and are narrowed on the device.
static void upload_index_array(const i64* h_src, size_t n, u32* d_dst, i64 lo, i64 hi, u32* d_flags) {
  if (n == 0) return;
  // (pinned sources take the same path: narrowing halves the bus bytes, and measured on C3 -- 2.2 GB of Int64 indices --
  //  the packed upload of PAGEABLE arrays, 31 ms, beats the plain DMA of pinned ones, 41 ms)
  if (n < PACK_CHUNK_ELEMS || staging_disabled() || std::getenv("CPB_NO_HOST_PACK")) {
    DBuf<i64> wide(n);
    h2d_copy(wide.get(), h_src, n * sizeof(i64));
    narrow_minus1(wide.get(), d_dst, n, lo, hi, d_flags);
    return;
  }
  uint64_t acc = 0;
  static const size_t chunk_elems = [] {  // (CPB_PACK_CHUNK: elements per staged chunk, for measurements; at most what a staging buffer holds)
    const char* e = std::getenv("CPB_PACK_CHUNK");
    const size_t v = e ? (size_t)std::atoll(e) : PACK_CHUNK_ELEMS;
    return std::min(std::max(v, (size_t)1 << 16), H2D_CHUNK / sizeof(u32));
  }();
  for (size_t off = 0; off < n; off += chunk_elems) {
    const int b = stage_acquire();
    const size_t cnt = std::min(chunk_elems, n - off);
    acc |= host_pack((uint32_t*)g_stage[b], reinterpret_cast<const int64_t*>(h_src + off), cnt);
    CPB_CUDA(cudaMemcpyAsync(d_dst + off, g_stage[b], cnt * sizeof(u32), cudaMemcpyHostToDevice, ctx().stream));
    stage_release(b);
    dec_check_u32(d_dst + off, cnt, lo, hi, d_flags);
  }
  CPB_REQUIRE((acc >> 31) == 0, "colptr/rowval entry out of range (expected 1-based indices below 2^31)");
}

extern "C++" {
template <class Ti> static void matrix_from_device(Matrix& M, i64 m, i64 n, i64 nnz, const Ti* d_colptr, const Ti* d_rowval) {
  CPB_REQUIRE(m >= 0 && n >= 0 && nnz >= 0, "negative dimension");
  CPB_REQUIRE(nnz + n + 1 < ((i64)1 << 31) && m < ((i64)1 << 31) - 2 && n < ((i64)1 << 31) - 2, "matrix too large for the 32-bit device index");
  M.m = m; M.n = n; M.N = nnz;
  M.pos.alloc((size_t)n + 1);
  M.row.alloc((size_t)nnz);
  DBuf<u32> flags(1);
  flags.zero();
  if constexpr (sizeof(Ti) == 8) {
    narrow_minus1((const i64*)d_colptr, M.pos.get(), (size_t)n + 1, 1, nnz + 1, flags.get());
    narrow_minus1((const i64*)d_rowval, M.row.get(), (size_t)nnz, 1, m, flags.get());
  } else {
    narrow32_minus1((const int*)d_colptr, M.pos.get(), (size_t)n + 1, 1, nnz + 1, flags.get());
    narrow32_minus1((const int*)d_rowval, M.row.get(), (size_t)nnz, 1, m, flags.get());
  }
  check_monotone(M.pos.get(), (size_t)n + 1, flags.get());
  u32 hf = 0;
  Ti ends[2] = {0, 0};
  CPB_CUDA(cudaMemcpyAsync(&hf, flags.get(), sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaMemcpyAsync(&ends[0], d_colptr, sizeof(Ti), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaMemcpyAsync(&ends[1], d_colptr + n, sizeof(Ti), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  CPB_REQUIRE((hf & 1u) == 0, "colptr/rowval entry out of range (expected 1-based indices)");
  CPB_REQUIRE((hf & 2u) == 0, "colptr is not non-decreasing");
  CPB_REQUIRE((i64)ends[0] == 1 && (i64)ends[1] == nnz + 1, "colptr[1] must be 1 and colptr[n+1] must be nnz+1");
}
}  // extern "C++"

int cpb_matrix_create_device(int64_t m, int64_t n, int64_t nnz, const int64_t* d_colptr, const int64_t* d_rowval, cpb_matrix** out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(out && d_colptr && (d_rowval || nnz == 0), "NULL argument");
  auto h = std::make_unique<cpb_matrix>();
  matrix_from_device(h->M, m, n, nnz, (const i64*)d_colptr, (const i64*)d_rowval);
  *out = h.release();
  CPB_API_END
}

int cpb_matrix_create(int64_t m, int64_t n, int64_t nnz, const int64_t* colptr, const int64_t* rowval, cpb_matrix** out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(out && colptr && (rowval || nnz == 0), "NULL argument");
  CPB_REQUIRE(m >= 0 && n >= 0 && nnz >= 0, "negative dimension");
  CPB_REQUIRE(nnz + n + 1 < ((i64)1 << 31) && m < ((i64)1 << 31) - 2 && n < ((i64)1 << 31) - 2, "matrix too large for the 32-bit device index");
  ProfScope prof("h2d_matrix", (double)(nnz + n + 1) * 8.0);
  auto h = std::make_unique<cpb_matrix>();
  Matrix& M = h->M;
  M.m = m; M.n = n; M.N = nnz;
  M.pos.alloc((size_t)n + 1);
  M.row.alloc((size_t)nnz);
  DBuf<u32> flags(1);
  flags.zero();
  upload_index_array((const i64*)colptr, (size_t)n + 1, M.pos.get(), 1, nnz + 1, flags.get());
  upload_index_array((const i64*)rowval, (size_t)nnz, M.row.get(), 1, m, flags.get());
  check_monotone(M.pos.get(), (size_t)n + 1, flags.get());
  u32 hf = 0;
  CPB_CUDA(cudaMemcpyAsync(&hf, flags.get(), sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  CPB_REQUIRE((hf & 1u) == 0, "colptr/rowval entry out of range (expected 1-based indices)");
  CPB_REQUIRE((hf & 2u) == 0, "colptr is not non-decreasing");
  CPB_REQUIRE(colptr[0] == 1 && colptr[n] == nnz + 1, "colptr[1] must be 1 and colptr[n+1] must be nnz+1");
  *out = h.release();
  CPB_API_END
}

int cpb_matrix_create_i32(int64_t m, int64_t n, int64_t nnz, const int32_t* colptr, const int32_t* rowval, cpb_matrix** out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(out && colptr && (rowval || nnz == 0), "NULL argument");
  CPB_REQUIRE(m >= 0 && n >= 0 && nnz >= 0, "negative dimension");
  ProfScope prof("h2d_matrix", (double)(nnz + n + 1) * 4.0);
  DBuf<int> dc((size_t)n + 1), dr((size_t)nnz);
  h2d_copy(dc.get(), colptr, ((size_t)n + 1) * sizeof(int));
  h2d_copy(dr.get(), rowval, (size_t)nnz * sizeof(int));
  auto h = std::make_unique<cpb_matrix>();
  matrix_from_device<int>(h->M, m, n, nnz, dc.get(), dr.get());
  *out = h.release();
  CPB_API_END
}

int cpb_matrix_dims(const cpb_matrix* A, int64_t* m, int64_t* n, int64_t* nnz) {
  CPB_API_BEGIN
  CPB_REQUIRE(A, "NULL matrix");
  if (m) *m = A->M.m;
  if (n) *n = A->M.n;
  if (nnz) *nnz = A->M.N;
  CPB_API_END
}

int cpb_matrix_get(const cpb_matrix* A, int64_t* colptr_out, int64_t* rowval_out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(A && colptr_out && (rowval_out || A->M.N == 0), "NULL argument");
  const Matrix& M = A->M;
  DBuf<i64> dc((size_t)M.n + 1), dr((size_t)M.N);
  widen_plus(M.pos.get(), dc.get(), (size_t)M.n + 1, 1);
  widen_plus(M.row.get(), dr.get(), (size_t)M.N, 1);
  CPB_CUDA(cudaMemcpyAsync(colptr_out, dc.get(), ((size_t)M.n + 1) * sizeof(i64), cudaMemcpyDeviceToHost, ctx().stream));
  if (M.N) CPB_CUDA(cudaMemcpyAsync(rowval_out, dr.get(), (size_t)M.N * sizeof(i64), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  CPB_API_END
}

void cpb_matrix_destroy(cpb_matrix* A) {
  std::lock_guard<std::mutex> lk(cpb::g_mu);
  if (cpb::g_ctx.ready) cudaSetDevice(cpb::g_ctx.device);
  delete A;
}

int cpb_adjointpattern(cpb_matrix* A, cpb_matrix** out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(A && out, "NULL argument");
  auto B = adjoint_pattern(A->M);
  auto h = std::make_unique<cpb_matrix>();
  h->M = std::move(*B);
  *out = h.release();
  CPB_API_END
}

int cpb_matrix_permute(cpb_matrix* A, const int64_t* col_prm, const int64_t* row_new, cpb_matrix** out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(A && out, "NULL argument");
  const Matrix& M = A->M;
  DBuf<u32> dc, dr, flags(1);
  flags.zero();
  auto upload = [&](const int64_t* h, i64 len, DBuf<u32>& d) {
    if (!h) return;
    DBuf<i64> wide((size_t)std::max<i64>(len, 1));
    h2d_copy(wide.get(), h, (size_t)len * sizeof(i64));
    d.alloc((size_t)std::max<i64>(len, 1));
    narrow_minus1(wide.get(), d.get(), (size_t)len, 1, len, flags.get());
  };
  upload(col_prm, M.n, dc);
  upload(row_new, M.m, dr);
  u32 hf = 0;
  CPB_CUDA(cudaMemcpyAsync(&hf, flags.get(), sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  CPB_REQUIRE(hf == 0, "permutation entry out of range (expected 1-based indices)");
  auto B = permute_pattern(M, col_prm ? dc.get() : nullptr, row_new ? dr.get() : nullptr);
  auto h = std::make_unique<cpb_matrix>();
  h->M = std::move(*B);
  *out = h.release();
  CPB_API_END
}

int cpb_oracle_create(cpb_matrix* A, const cpb_model* mdl, const int64_t* pi_spl, int64_t pi_K, cpb_oracle** out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(A && mdl && out, "NULL argument");
  trace_mark("enter");
  auto h = std::make_unique<cpb_oracle>();
  h->O = oracle_create(A->M, mdl, pi_spl, pi_K);
  *out = h.release();
  trace_mark("exit");
  trace_flush("oracle_create");
  CPB_API_END
}

void cpb_oracle_destroy(cpb_oracle* f) {
  std::lock_guard<std::mutex> lk(cpb::g_mu);
  if (cpb::g_ctx.ready) cudaSetDevice(cpb::g_ctx.device);
  delete f;
}

int cpb_oracle_query_device(cpb_oracle* f, int64_t Q, const int64_t* d_j, const int64_t* d_jp, double* d_cost_out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(f && (Q == 0 || (d_j && d_jp && d_cost_out)), "NULL argument");
  if (f->O->mdl.kind >= CPB_MODEL_PRIMCONN && f->O->mdl.kind <= CPB_MODEL_SECEDGE)
    // (this entry point carries no part index: the row-partition-aware oracles would silently answer for part 1 -- ADVICE r1)
    throw Error(CPB_ERR_UNSUPPORTED, "cpb_oracle_query_device has no part index: use cpb_oracle_query for the row-partition-aware models");
  oracle_query(*f->O, Q, (const i64*)d_j, (const i64*)d_jp, d_cost_out);
  CPB_API_END
}

int cpb_oracle_query(cpb_oracle* f, int64_t Q, const int64_t* j, const int64_t* jp, const int64_t* k, double* cost_out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(f && Q >= 0 && (Q == 0 || (j && jp && cost_out)), "NULL argument");
  if (Q > 0) {
    const i64 n1 = f->O->A->n + 1;
    for (i64 t = 0; t < Q; ++t) CPB_REQUIRE(j[t] >= 1 && jp[t] >= j[t] && jp[t] <= n1, "query out of range (need 1 <= j <= j' <= n+1)");
    DBuf<i64> dj(Q), djp(Q), dk(k ? Q : 0);
    DBuf<double> dc(Q);
    CPB_CUDA(cudaMemcpyAsync(dj.get(), j, Q * sizeof(i64), cudaMemcpyHostToDevice, ctx().stream));
    CPB_CUDA(cudaMemcpyAsync(djp.get(), jp, Q * sizeof(i64), cudaMemcpyHostToDevice, ctx().stream));
    if (k) CPB_CUDA(cudaMemcpyAsync(dk.get(), k, Q * sizeof(i64), cudaMemcpyHostToDevice, ctx().stream));  // part index (1-based): only the row-partition-aware models use it
    oracle_query(*f->O, Q, dj.get(), djp.get(), dc.get(), k ? dk.get() : nullptr);
    CPB_CUDA(cudaMemcpyAsync(cost_out, dc.get(), Q * sizeof(double), cudaMemcpyDeviceToHost, ctx().stream));
    CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  }
  CPB_API_END
}

int cpb_count_query(cpb_matrix* A, int which, int64_t Q, const int64_t* j, const int64_t* jp, int64_t* out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(A && Q >= 0 && (Q == 0 || (j && jp && out)), "NULL argument");
  const i64 n1 = A->M.n + 1;
  for (i64 t = 0; t < Q; ++t) CPB_REQUIRE(j[t] >= 1 && jp[t] >= j[t] && jp[t] <= n1, "query out of range (need 1 <= j <= j' <= n+1)");
  DBuf<i64> dj(Q), djp(Q), dout(Q);
  if (Q) {
    CPB_CUDA(cudaMemcpyAsync(dj.get(), j, Q * sizeof(i64), cudaMemcpyHostToDevice, ctx().stream));
    CPB_CUDA(cudaMemcpyAsync(djp.get(), jp, Q * sizeof(i64), cudaMemcpyHostToDevice, ctx().stream));
  }
  count_query(A->M, which, Q, dj.get(), djp.get(), dout.get());
  if (Q) CPB_CUDA(cudaMemcpyAsync(out, dout.get(), Q * sizeof(i64), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  CPB_API_END
}

int cpb_prefix_create(int64_t m, int64_t n, int64_t N, const int64_t* pos, const int64_t* idx, const int64_t* val, cpb_prefix** out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(out && (idx || N == 0), "NULL argument");
  CPB_REQUIRE(m >= 0 && n >= 0 && N >= 0, "negative dimension");
  DBuf<i64> dpos(pos ? (size_t)n + 1 : 0), didx((size_t)std::max<int64_t>(N, 1)), dval(val ? (size_t)std::max<int64_t>(N, 1) : 0);
  if (pos) h2d_copy(dpos.get(), pos, ((size_t)n + 1) * sizeof(i64));
  h2d_copy(didx.get(), idx, (size_t)N * sizeof(i64));
  if (val) h2d_copy(dval.get(), val, (size_t)N * sizeof(i64));
  auto h = std::make_unique<cpb_prefix>();
  h->P = prefix_build(m, n, N, pos ? dpos.get() : nullptr, didx.get(), val ? dval.get() : nullptr);
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  *out = h.release();
  CPB_API_END
}

int cpb_prefix_query(cpb_prefix* P, int64_t Q, const int64_t* i, const int64_t* j, int64_t* count_out, int64_t* sum_out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(P && Q >= 0 && (Q == 0 || (i && j)), "NULL argument");
  const PrefixMatrix& M = *P->P;
  for (i64 t = 0; t < Q; ++t) CPB_REQUIRE(i[t] >= 1 && i[t] <= M.m + 1 && j[t] >= 1 && j[t] <= M.n + 1, "index out of range (need 1 <= i <= m+1, 1 <= j <= n+1)");
  DBuf<i64> di(Q), dj(Q), dc(count_out ? Q : 0), ds(sum_out ? Q : 0);
  if (Q) {
    CPB_CUDA(cudaMemcpyAsync(di.get(), i, Q * sizeof(i64), cudaMemcpyHostToDevice, ctx().stream));
    CPB_CUDA(cudaMemcpyAsync(dj.get(), j, Q * sizeof(i64), cudaMemcpyHostToDevice, ctx().stream));
  }
  prefix_query(M, Q, di.get(), dj.get(), count_out ? dc.get() : nullptr, sum_out ? ds.get() : nullptr);
  if (Q && count_out) CPB_CUDA(cudaMemcpyAsync(count_out, dc.get(), Q * sizeof(i64), cudaMemcpyDeviceToHost, ctx().stream));
  if (Q && sum_out) CPB_CUDA(cudaMemcpyAsync(sum_out, ds.get(), Q * sizeof(i64), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  CPB_API_END
}

void cpb_prefix_destroy(cpb_prefix* P) {
  std::lock_guard<std::mutex> lk(cpb::g_mu);
  if (cpb::g_ctx.ready) cudaSetDevice(cpb::g_ctx.device);
  delete P;
}

int cpb_bound_stripe(cpb_oracle* f, int64_t K, double out[2]) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(f && out, "NULL argument");
  oracle_bound(*f->O, K, out);
  CPB_API_END
}

int cpb_objective(cpb_oracle* f, int total, int64_t K, const int64_t* spl, double* out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(f && spl && out, "NULL argument");
  *out = oracle_objective(*f->O, total != 0, K, spl);
  CPB_API_END
}

// partition_stripe's method dispatch (the caller holds the library lock)
static void partition_stripe_impl(cpb_oracle* f, int method, const cpb_constraint* con, double eps, int64_t K, int64_t* spl_out) {
  if ((method == CPB_SPLIT_DYNAMIC_BOTTLENECK_CHUNKER || method == CPB_SPLIT_DYNAMIC_TOTAL_CHUNKER) && f->O->mdl.kind >= CPB_MODEL_PRIMCONN &&
      f->O->mdl.kind <= CPB_MODEL_SECEDGE)
    // the chunker-form K-DP calls f(j, j') without a part index (DynamicSplitter.jl:62-71, 290-301): a MethodError for the
    // partition-aware oracles, whose only method is (j, j', k) (PrimaryConnectivityCosts.jl:66, SecondaryConnectivityCosts.jl:82, ...)
    throw Error(CPB_ERR_UNSUPPORTED, "the chunker-form K-DP has no method for the row-partition-aware cost models (the reference calls f(j, j') without k)");
  switch (method) {
    case CPB_SPLIT_DYNAMIC_BOTTLENECK: case CPB_SPLIT_DYNAMIC_BOTTLENECK_CHUNKER: solve_dynamic(*f->O, false, con, K, spl_out); break;
    case CPB_SPLIT_DYNAMIC_TOTAL: case CPB_SPLIT_DYNAMIC_TOTAL_CHUNKER: solve_dynamic(*f->O, true, con, K, spl_out); break;
    case CPB_SPLIT_CONVEX_TOTAL: solve_convex_splitter(*f->O, con, K, spl_out); break;
    case CPB_SPLIT_CONCAVE_TOTAL: solve_concave_splitter(*f->O, con, K, spl_out); break;
    case CPB_SPLIT_BISECT_COST: solve_bisect(*f->O, false, eps, K, spl_out); break;
    case CPB_SPLIT_LAZY_BISECT_COST: solve_bisect(*f->O, true, eps, K, spl_out); break;
    case CPB_SPLIT_BISECT_INDEX: solve_bisect_index(*f->O, K, spl_out); break;
    case CPB_SPLIT_FLIP_BISECT_COST: case CPB_SPLIT_LAZY_FLIP_BISECT_COST: case CPB_SPLIT_FLIP_BISECT_INDEX:
      solve_flip(*f->O, method, eps, K, spl_out);
      break;
    case CPB_SPLIT_EQUI: {  // EquiPartitioner.jl:3-9
      const i64 n = f->O->A->n;
      for (i64 k = 1; k <= K + 1; ++k) spl_out[k - 1] = (k - 1) * (n / K) + std::min(n % K, k - 1) + 1;
      break;
    }
    default: throw Error(CPB_ERR_UNSUPPORTED, "unsupported partition_stripe method");
  }
}

int cpb_partition_stripe(cpb_oracle* f, int method, const cpb_constraint* con, double eps, int64_t K, int64_t* spl_out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(f && spl_out, "NULL argument");
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  trace_mark("enter");
  struct TraceEnd { ~TraceEnd() { trace_mark("exit"); trace_flush("partition_stripe"); } } trace_end;
  partition_stripe_impl(f, method, con, eps, K, spl_out);
  CPB_API_END
}

int cpb_partition_stripe_batch(int64_t B, cpb_oracle* const* f, const int* method, const double* eps, const int64_t* K, int64_t* const* spl_out) {
  CPB_API_BEGIN
  CPB_REQUIRE(B >= 0, "B must be >= 0");
  if (B == 0) return CPB_OK;
  ensure_context();
  CPB_REQUIRE(f && method && K && spl_out, "NULL argument");
  std::vector<Oracle*> O(B);
  for (int64_t b = 0; b < B; ++b) {
    if (!f[b]) throw Error(CPB_ERR_ARG, "problem " + std::to_string(b) + ": NULL argument");
    O[b] = f[b]->O.get();
  }
  trace_mark("enter");
  struct TraceEnd { ~TraceEnd() { trace_mark("exit"); trace_flush("partition_stripe_batch"); } } trace_end;
  solve_stripe_batch(B, O.data(), method, eps, (const i64*)K, spl_out);
  CPB_API_END
}

int cpb_partition_stripe_batch_capacity(int* clusters_out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(clusters_out, "NULL argument");
  *clusters_out = stripe_batch_capacity();
  CPB_API_END
}

int cpb_partition_stripe_weighted(cpb_oracle* f, int method, cpb_oracle* w, int64_t w_max, double eps, int64_t K, int64_t* spl_out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(f && w && spl_out, "NULL argument");
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  CPB_REQUIRE(f->O->A == w->O->A, "the weight oracle must be built on the same cpb_matrix as the cost oracle");
  trace_mark("enter");
  struct TraceEnd { ~TraceEnd() { trace_mark("exit"); trace_flush("partition_stripe_weighted"); } } trace_end;
  if (method != CPB_SPLIT_DYNAMIC_BOTTLENECK && method != CPB_SPLIT_DYNAMIC_TOTAL && method != CPB_SPLIT_DYNAMIC_BOTTLENECK_CHUNKER &&
      method != CPB_SPLIT_DYNAMIC_TOTAL_CHUNKER && method != CPB_SPLIT_CONVEX_TOTAL && method != CPB_SPLIT_CONCAVE_TOTAL)
    throw Error(CPB_ERR_UNSUPPORTED, "a weight constraint is taken by the Dynamic, Convex and Concave total splitters only");
  weight_check(*w->O);
  if (w->O->mdl.kind == CPB_MODEL_WORK) {  // an affine work weight: the cpb_constraint path, one implementation of its windows
    cpb_constraint con{};
    con.enabled = 1;
    for (int t = 0; t < 3; ++t) con.w_coef[t] = (int64_t)w->O->mdl.coef[t];
    con.w_max = w_max;
    partition_stripe_impl(f, method, &con, eps, K, spl_out);
    return CPB_OK;
  }
  if ((method == CPB_SPLIT_DYNAMIC_BOTTLENECK_CHUNKER || method == CPB_SPLIT_DYNAMIC_TOTAL_CHUNKER) && f->O->mdl.kind >= CPB_MODEL_PRIMCONN &&
      f->O->mdl.kind <= CPB_MODEL_SECEDGE)
    throw Error(CPB_ERR_UNSUPPORTED, "the chunker-form K-DP has no method for the row-partition-aware cost models (the reference calls f(j, j') without k)");
  switch (method) {
    case CPB_SPLIT_DYNAMIC_BOTTLENECK: case CPB_SPLIT_DYNAMIC_BOTTLENECK_CHUNKER: solve_dynamic_weighted(*f->O, false, *w->O, w_max, K, spl_out); break;
    case CPB_SPLIT_DYNAMIC_TOTAL: case CPB_SPLIT_DYNAMIC_TOTAL_CHUNKER: solve_dynamic_weighted(*f->O, true, *w->O, w_max, K, spl_out); break;
    case CPB_SPLIT_CONVEX_TOTAL: solve_convex_weighted(*f->O, *w->O, w_max, K, spl_out); break;
    case CPB_SPLIT_CONCAVE_TOTAL: solve_concave_weighted(*f->O, *w->O, w_max, K, spl_out); break;
    default: throw Error(CPB_ERR_UNSUPPORTED, "a weight constraint is taken by the Dynamic, Convex and Concave total splitters only");
  }
  CPB_API_END
}

int cpb_weight_windows(cpb_oracle* w, int64_t w_max, int64_t* first_fit_out, int64_t* reach_out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(w && first_fit_out && reach_out, "NULL argument");
  DBuf<u32> ff, rc;
  weight_windows(*w->O, w_max, ff, &rc);
  const size_t n1 = (size_t)w->O->A->n + 1;
  std::vector<u32> h(2 * n1);
  CPB_CUDA(cudaMemcpyAsync(h.data(), ff.get() + 1, n1 * sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaMemcpyAsync(h.data() + n1, rc.get() + 1, n1 * sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  for (size_t c = 0; c < n1; ++c) {
    first_fit_out[c] = h[c];
    reach_out[c] = h[n1 + c];
  }
  CPB_API_END
}

int cpb_bisect_plan(double c_lo, double c_hi, double eps, int nodes, double c_lo0, double c_hi0, double upper_bound, int32_t* ids_out) {
  CPB_API_BEGIN
  CPB_REQUIRE(ids_out && nodes >= 1 && nodes <= 255, "bad plan request");
  bisect_plan_nodes(c_lo, c_hi, eps, nodes, c_lo0, c_hi0, upper_bound, true, ids_out);
  CPB_API_END
}

int cpb_bisect_prewalk(double c_lo, double c_hi, double eps, double upper_bound, double* c_hi_out, int32_t* probes_out) {
  CPB_API_BEGIN
  CPB_REQUIRE(c_hi_out && probes_out, "NULL argument");
  int probes = 0;
  bisect_prewalk(c_lo, c_hi, eps, upper_bound, c_hi_out, &probes);
  *probes_out = probes;
  CPB_API_END
}

int cpb_bisect_stats(double out[8]) {
  CPB_API_BEGIN
  CPB_REQUIRE(out, "NULL argument");
  bisect_stats(out);
  CPB_API_END
}

// ---- multi-GPU: library-owned communicator, one solve over all ranks (sharded.cu) ----
extern "C++" {
namespace cpb {
struct ShardedMatrix;
void comm_unique_id(char out[128]);
void comm_init(const char id[128], int rank, int world);
void comm_destroy();
void comm_info(int* rank, int* world);
void shard_range(i64 N, int rank, int world, i64* cnt_out, i64* lo_out, i64* hi_out);
ShardedMatrix* sharded_create(i64 m, i64 n, i64 nnz, const i64* h_colptr, const i64* h_rowval, bool rows_are_block,
                              void (*upload)(const i64*, size_t, u32*, i64, i64, u32*));
void sharded_destroy(ShardedMatrix* S);
void solve_sharded(ShardedMatrix& S, const cpb_model* mdl, int method, double eps, i64 K, int64_t* h_spl_out);
void solve_sharded_emulated(Matrix& A, const cpb_model* mdl, int method, double eps, i64 K, int world, int64_t* h_spl_out);
void sharded_stats(double out[16]);
ShardedMatrix* sharded_adjointpattern(const ShardedMatrix& S);
std::unique_ptr<Matrix> adjoint_pattern_sharded_emulated(const Matrix& A, int world);
void sharded_dims(const ShardedMatrix& S, i64* m, i64* n, i64* nnz, i64* q_lo, i64* q_hi);
void sharded_get(const ShardedMatrix& S, i64* h_colptr, i64* h_rowval_blk);
}  // namespace cpb
}  // extern "C++"

int cpb_comm_unique_id(char id_out[128]) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(id_out, "NULL argument");
  comm_unique_id(id_out);
  CPB_API_END
}
int cpb_comm_init(const char id[128], int rank, int world) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(id, "NULL argument");
  comm_init(id, rank, world);
  CPB_API_END
}
int cpb_comm_destroy(void) {
  CPB_API_BEGIN
  if (cpb::g_ctx.ready) { CPB_CUDA(cudaSetDevice(cpb::g_ctx.device)); comm_destroy(); }
  CPB_API_END
}
int cpb_comm_info(int* rank, int* world) {
  CPB_API_BEGIN
  comm_info(rank, world);
  CPB_API_END
}
int cpb_shard_range(int64_t nnz, int rank, int world, int64_t* q_lo, int64_t* q_hi) {
  CPB_API_BEGIN
  CPB_REQUIRE(world >= 1 && rank >= 0 && rank < world && nnz >= 0, "bad shard request");
  i64 lo = 0, hi = 0;
  shard_range(nnz, rank, world, nullptr, &lo, &hi);
  if (q_lo) *q_lo = lo;
  if (q_hi) *q_hi = hi;
  CPB_API_END
}
int cpb_sharded_matrix_create(int64_t m, int64_t n, int64_t nnz, const int64_t* colptr, const int64_t* rowval, int rowval_is_block, cpb_sharded** out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(out && colptr && (rowval || nnz == 0), "NULL argument");
  ProfScope prof("h2d_matrix");
  *out = reinterpret_cast<cpb_sharded*>(sharded_create(m, n, nnz, (const i64*)colptr, (const i64*)rowval, rowval_is_block != 0, upload_index_array));
  CPB_API_END
}
void cpb_sharded_matrix_destroy(cpb_sharded* A) {
  std::lock_guard<std::mutex> lk(cpb::g_mu);
  if (cpb::g_ctx.ready) cudaSetDevice(cpb::g_ctx.device);
  sharded_destroy(reinterpret_cast<ShardedMatrix*>(A));
}
int cpb_partition_stripe_sharded(cpb_sharded* A, const cpb_model* mdl, int method, double eps, int64_t K, int64_t* spl_out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(A && mdl && spl_out, "NULL argument");
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  solve_sharded(*reinterpret_cast<ShardedMatrix*>(A), mdl, method, eps, K, spl_out);
  CPB_API_END
}
int cpb_partition_stripe_sharded_emulated(cpb_matrix* A, const cpb_model* mdl, int method, double eps, int64_t K, int world, int64_t* spl_out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(A && mdl && spl_out, "NULL argument");
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  solve_sharded_emulated(A->M, mdl, method, eps, K, world, spl_out);
  CPB_API_END
}
int cpb_sharded_adjointpattern(cpb_sharded* A, cpb_sharded** out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(A && out, "NULL argument");
  *out = reinterpret_cast<cpb_sharded*>(sharded_adjointpattern(*reinterpret_cast<ShardedMatrix*>(A)));
  CPB_API_END
}
int cpb_adjointpattern_sharded_emulated(cpb_matrix* A, int world, cpb_matrix** out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(A && out, "NULL argument");
  auto B = adjoint_pattern_sharded_emulated(A->M, world);
  auto h = std::make_unique<cpb_matrix>();
  h->M = std::move(*B);
  *out = h.release();
  CPB_API_END
}
int cpb_sharded_matrix_get(const cpb_sharded* A, int64_t* colptr_out, int64_t* rowval_block_out, int64_t* q_lo, int64_t* q_hi) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(A, "NULL argument");
  const ShardedMatrix& S = *reinterpret_cast<const ShardedMatrix*>(A);
  i64 lo = 0, hi = 0;
  sharded_dims(S, nullptr, nullptr, nullptr, &lo, &hi);
  if (q_lo) *q_lo = lo;
  if (q_hi) *q_hi = hi;
  if (colptr_out || rowval_block_out) sharded_get(S, (i64*)colptr_out, (i64*)rowval_block_out);
  CPB_API_END
}
int cpb_sharded_stats(double out[16]) {
  CPB_API_BEGIN
  CPB_REQUIRE(out, "NULL argument");
  sharded_stats(out);
  CPB_API_END
}

int cpb_pack_stripe(cpb_matrix* A, cpb_oracle* f, int method, const cpb_constraint* con, double rho, int64_t w_max,
                    int64_t* spl_out, int64_t* K_out, int64_t* n_nets_out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(A && spl_out && K_out, "NULL argument");
  trace_mark("enter");
  struct TraceEnd { ~TraceEnd() { trace_mark("exit"); trace_flush("pack_stripe"); } } trace_end;
  solve_pack(A->M, f ? f->O.get() : nullptr, method, con, rho, w_max, spl_out, K_out, n_nets_out);
  CPB_API_END
}

int cpb_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(cpb::g_mu);
  cpb::g_ctx.profiling = on != 0;
  return CPB_OK;
}

int cpb_profile_reset(void) {
  std::lock_guard<std::mutex> lk(cpb::g_mu);
  if (cpb::g_ctx.ready) cpb::resolve_pending();
  cpb::g_ctx.prof.clear();
  cpb::g_ctx.launches = 0;
  return CPB_OK;
}

int cpb_profile_get(int cap, char* names, double* ms, int64_t* launches, double* bytes) {
  std::lock_guard<std::mutex> lk(cpb::g_mu);
  if (cpb::g_ctx.ready) cpb::resolve_pending();
  int k = 0;
  for (auto& p : cpb::g_ctx.prof) {
    if (k >= cap) break;
    std::memset(names + 32 * k, 0, 32);
    std::strncpy(names + 32 * k, p.first.c_str(), 31);
    ms[k] = p.second.ms;
    launches[k] = p.second.launches;
    bytes[k] = p.second.bytes;
    ++k;
  }
  return k;
}

int64_t cpb_launch_count(void) { return cpb::g_ctx.launches; }

static cudaEvent_t g_t0 = nullptr, g_t1 = nullptr;
int cpb_timer_start(void) {
  CPB_API_BEGIN
  ensure_context();
  if (!g_t0) { CPB_CUDA(cudaEventCreate(&g_t0)); CPB_CUDA(cudaEventCreate(&g_t1)); }
  CPB_CUDA(cudaEventRecord(g_t0, ctx().stream));
  CPB_API_END
}
int cpb_timer_stop(double* ms_out) {
  CPB_API_BEGIN
  ensure_context();
  CPB_REQUIRE(g_t0 && ms_out, "timer not started");
  CPB_CUDA(cudaEventRecord(g_t1, ctx().stream));
  CPB_CUDA(cudaEventSynchronize(g_t1));
  float ms = 0;
  CPB_CUDA(cudaEventElapsedTime(&ms, g_t0, g_t1));
  *ms_out = ms;
  CPB_API_END
}

}  // extern "C"
