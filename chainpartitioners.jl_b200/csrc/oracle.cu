// oracle.cu -- oracle_stripe on the device: builds the structures a cost model needs and answers
// batched c(j, j', k) queries (kernel "oracle_query_batch"), bound_stripe and objective values.
#include <algorithm>
#include <cmath>
#include "engine.cuh"
#include "primitives.cuh"

namespace cpb {

static unsigned grid_for(size_t n) { return (unsigned)std::max<size_t>(1, std::min<size_t>((n + 255) / 256, (size_t)ctx().sm_count * 32)); }

// ---- Julia's fld (Base div.jl) on the host, for bound_stripe ------------------------------------
static i64 jl_fld(i64 x, i64 y) {
  i64 q = x / y, r = x % y;
  if (r != 0 && ((r < 0) != (y < 0))) q -= 1;
  return q;
}
static double jl_mod(double x, double y) {
  double r = std::fmod(x, y);
  if (r == 0) return std::copysign(r, y);
  if ((r > 0) != (y > 0)) return r + y;
  return r;
}
static double jl_fld(double x, double y) { return std::nearbyint((x - jl_mod(x, y)) / y); }

// ---- structure kernels --------------------------------------------------------------------------
__global__ void k_overdeg(const u32* __restrict__ pos, u32 n, i64 delta, u32* __restrict__ out) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j <= n; j += stride) {
    i64 v = 0;
    if (j < n) v = max((i64)(pos[j + 1] - pos[j]) - delta, (i64)0);
    out[j] = (u32)v;
  }
}

__global__ void k_env_leaves(const u32* __restrict__ pos, const u32* __restrict__ row, u32 n, u32 m, int H, i64* __restrict__ tree) {
  const size_t leaves = (size_t)1 << H;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < leaves; t += stride) {
    i64 lo = (i64)m + 1, hi = 0;
    if (t < n && pos[t] < pos[t + 1]) {
      lo = (i64)row[pos[t]] + 1;
      hi = (i64)row[pos[t + 1] - 1] + 1;
    }
    tree[leaves + t] = (lo << 32) | hi;  // 1-based node (2^H - 1) + (t + 1)
  }
}
__global__ void k_env_level(i64* __restrict__ tree, size_t first, size_t count) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < count; t += stride) {
    const size_t i = first + t;
    const i64 l = tree[2 * i], r = tree[2 * i + 1];
    tree[i] = (min(l >> 32, r >> 32) << 32) | max(l & 0xffffffffll, r & 0xffffffffll);
  }
}

__global__ void k_row_extrema(const u32* __restrict__ row, size_t N, u32* __restrict__ out /* [0]=min, [1]=max */) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  u32 lo = 0xffffffffu, hi = 0;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < N; q += stride) {
    lo = min(lo, row[q]);
    hi = max(hi, row[q]);
  }
  for (int o = 16; o > 0; o >>= 1) {
    lo = min(lo, __shfl_down_sync(0xffffffffu, lo, o));
    hi = max(hi, __shfl_down_sync(0xffffffffu, hi, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMin(out, lo);
    atomicMax(out + 1, hi);
  }
}

__global__ void k_pi_assign(const u32* __restrict__ spl0 /* K+1, 0-based */, u32 K, u32* __restrict__ asg, u32* __restrict__ size) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < K; k += stride) {
    size[k] = spl0[k + 1] - spl0[k];
    for (u32 i = spl0[k]; i < spl0[k + 1]; ++i) asg[i] = (u32)k;
  }
}

std::unique_ptr<Oracle> oracle_create(Matrix& A, const cpb_model* mdl, const int64_t* pi_spl, i64 pi_K) {
  CPB_REQUIRE(mdl != nullptr, "model is NULL");
  auto f = std::make_unique<Oracle>();
  f->A = &A;
  f->mdl = *mdl;
  DevOracle& d = f->dev;
  std::memset(&d, 0, sizeof(d));
  d.kind = mdl->kind;
  d.is_float = mdl->is_float;
  d.n = (u32)A.n;
  d.m = (u32)A.m;
  d.pos = A.pos.get();
  for (int t = 0; t < 5; ++t) {
    d.cf[t] = mdl->coef[t];
    d.ci[t] = (i64)std::llround(mdl->coef[t]);
    if (!mdl->is_float) CPB_REQUIRE((double)d.ci[t] == mdl->coef[t], "Int64 model with a non-integer coefficient");
  }
  switch (mdl->kind) {
    case CPB_MODEL_WORK: break;
    case CPB_MODEL_CONNECTIVITY: break;
    case CPB_MODEL_COLBLOCK: {
      CPB_REQUIRE(mdl->alpha_col && mdl->beta_col && mdl->w_tab >= 0, "column-block model needs tables");
      const int W = mdl->w_tab + 1;
      std::vector<double> hf(2 * (size_t)W);
      std::vector<i64> hi(2 * (size_t)W);
      for (int w = 0; w < W; ++w) {
        hf[w] = mdl->alpha_col[w];
        hf[W + w] = mdl->beta_col[w];
        hi[w] = (i64)std::llround(hf[w]);
        hi[W + w] = (i64)std::llround(hf[W + w]);
      }
      f->tab_f.alloc(hf.size());
      f->tab_i.alloc(hi.size());
      CPB_CUDA(cudaMemcpyAsync(f->tab_f.get(), hf.data(), hf.size() * sizeof(double), cudaMemcpyHostToDevice, ctx().stream));
      CPB_CUDA(cudaMemcpyAsync(f->tab_i.get(), hi.data(), hi.size() * sizeof(i64), cudaMemcpyHostToDevice, ctx().stream));
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));  // host staging vectors die at scope exit
      d.tab_alpha_f = f->tab_f.get();
      d.tab_beta_f = f->tab_f.get() + W;
      d.tab_alpha_i = f->tab_i.get();
      d.tab_beta_i = f->tab_i.get() + W;
      d.w_tab = mdl->w_tab;
      f->h_alpha_col.assign(mdl->alpha_col, mdl->alpha_col + W);
      f->h_beta_col.assign(mdl->beta_col, mdl->beta_col + W);
      break;
    }
    case CPB_MODEL_MONOSYM: {
      CPB_REQUIRE(A.m == A.n, "monotonized symmetric model needs a square matrix");  // Monotonized...:80
      CPB_REQUIRE(mdl->coef[4] == std::floor(mdl->coef[4]), "delta_pins must be integer valued");
      f->overpos.alloc((size_t)A.n + 1);
      CPB_LAUNCH(k_overdeg, grid_for((size_t)A.n + 1), 256, 0, A.pos.get(), (u32)A.n, (i64)mdl->coef[4], f->overpos.get());
      exclusive_scan_u32(f->overpos.get(), f->overpos.get(), (size_t)A.n + 1);
      d.overpos = f->overpos.get();
      break;
    }
    case CPB_MODEL_SYMCONN:
      CPB_REQUIRE(A.m == A.n, "symmetric connectivity model needs a square matrix");  // Symmetric...:32
      break;
    case CPB_MODEL_HYPEREDGE: break;
    case CPB_MODEL_SYMEDGECUT: break;
    case CPB_MODEL_ENVELOPE: {
      int H = 0;
      while (((i64)1 << H) < std::max<i64>(A.n, 1)) ++H;  // cllog2(n)
      f->envH = H;
      const size_t leaves = (size_t)1 << H;
      f->env.alloc(2 * leaves);
      CPB_LAUNCH(k_env_leaves, grid_for(leaves), 256, 0, A.pos.get(), A.row.get(), (u32)A.n, (u32)A.m, H, f->env.get());
      for (int h = H - 1; h >= 0; --h) {
        const size_t first = (size_t)1 << h, count = (size_t)1 << h;
        CPB_LAUNCH(k_env_level, grid_for(count), 256, 0, f->env.get(), first, count);
      }
      d.env = f->env.get();
      d.envH = H;
      break;
    }
    case CPB_MODEL_PRIMEDGE:
    case CPB_MODEL_SECEDGE:
    case CPB_MODEL_SECCONN:
    case CPB_MODEL_PRIMCONN: {  // PrimaryConnectivityCosts.jl:56-67 / SecondaryConnectivityCosts.jl:67-81: need the row partition Pi
      CPB_REQUIRE(pi_spl != nullptr && pi_K >= 1, "primary / secondary connectivity models need a row partition (SplitPartition)");
      CPB_REQUIRE(pi_spl[0] == 1 && pi_spl[pi_K] == A.m + 1, "row partition must cover rows 1..m");
      f->pi_K = pi_K;
      f->h_pi_spl.assign(pi_spl, pi_spl + pi_K + 1);
      std::vector<u32> spl0(pi_K + 1);
      for (i64 k = 0; k <= pi_K; ++k) {
        CPB_REQUIRE(k == 0 || pi_spl[k] >= pi_spl[k - 1], "row partition must be sorted");
        spl0[k] = (u32)(pi_spl[k] - 1);
      }
      DBuf<u32> dspl(pi_K + 1);
      CPB_CUDA(cudaMemcpyAsync(dspl.get(), spl0.data(), spl0.size() * sizeof(u32), cudaMemcpyHostToDevice, ctx().stream));
      f->pi_asg.alloc((size_t)A.m);
      f->pi_size.alloc((size_t)pi_K);
      CPB_LAUNCH(k_pi_assign, grid_for((size_t)pi_K), 256, 0, dspl.get(), (u32)pi_K, f->pi_asg.get(), f->pi_size.get());
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));
      break;
    }
    case CPB_MODEL_BLOCK: {
      CPB_REQUIRE(pi_spl != nullptr && pi_K >= 0, "block cost model needs a row partition (SplitPartition)");
      CPB_REQUIRE(mdl->R >= 0 && mdl->R <= 4, "block model supports up to 4 components");
      CPB_REQUIRE(pi_spl[0] == 1 && pi_spl[pi_K] == A.m + 1, "row partition must cover rows 1..m");
      f->pi_K = pi_K;
      f->h_pi_spl.assign(pi_spl, pi_spl + pi_K + 1);
      std::vector<u32> spl0(pi_K + 1);
      for (i64 k = 0; k <= pi_K; ++k) {
        CPB_REQUIRE(k == 0 || pi_spl[k] >= pi_spl[k - 1], "row partition must be sorted");
        spl0[k] = (u32)(pi_spl[k] - 1);
      }
      DBuf<u32> dspl(pi_K + 1);
      CPB_CUDA(cudaMemcpyAsync(dspl.get(), spl0.data(), spl0.size() * sizeof(u32), cudaMemcpyHostToDevice, ctx().stream));
      f->pi_asg.alloc((size_t)A.m);
      f->pi_size.alloc((size_t)pi_K);
      if (pi_K) CPB_LAUNCH(k_pi_assign, grid_for((size_t)pi_K), 256, 0, dspl.get(), (u32)pi_K, f->pi_asg.get(), f->pi_size.get());
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));
      const int W = mdl->w_tab + 1, U = mdl->u_tab + 1;
      f->h_alpha_col.assign(mdl->alpha_col, mdl->alpha_col + W);
      f->h_beta_col.assign(mdl->beta_col, mdl->beta_col + (size_t)mdl->R * W);
      f->h_beta_row.assign(mdl->beta_row, mdl->beta_row + (size_t)mdl->R * U);
      break;
    }
    default: throw Error(CPB_ERR_UNSUPPORTED, "unknown cost model kind");
  }
  // the caller's table pointers are not retained (ABI contract): host copies live in the handle
  f->mdl.alpha_col = f->mdl.beta_col = f->mdl.beta_row = nullptr;
  return f;
}

// Builds the dominance indices the model's random-access oracle needs, on first use.  The chunkers
// (pack_stripe) never call this: they stream the link arrays instead.
void oracle_ensure_ranks(Oracle& f) {
  if (f.ranks_built) return;
  ProfScope prof("oracle_stripe");
  Matrix& A = *f.A;
  DevOracle& d = f.dev;
  switch (f.mdl.kind) {
    case CPB_MODEL_CONNECTIVITY: case CPB_MODEL_COLBLOCK: f.net = build_rank(A, RANK_NET); break;
    case CPB_MODEL_MONOSYM: f.dianet = build_rank(A, RANK_DIANET); break;
    case CPB_MODEL_SYMCONN: f.net = build_rank(A, RANK_NET); f.dianet = build_rank(A, RANK_DIANET); break;
    case CPB_MODEL_HYPEREDGE: f.net = build_rank(A, RANK_NET); f.selfnet = build_rank(A, RANK_SELFNET); break;
    case CPB_MODEL_SYMEDGECUT: f.selfpin = build_rank(A, RANK_SELFPIN); break;
    case CPB_MODEL_PRIMEDGE:
    case CPB_MODEL_SECEDGE:
    case CPB_MODEL_SECCONN:
      build_partwise_columns(A, f.pi_asg.get(), (u32)f.pi_K, f.part_col, f.part_start, f.part_head);
      d.part_col = f.part_col.get();
      d.part_start = f.part_start.get();
      d.part_head = f.part_head.get();
      d.part_size = f.pi_size.get();
      d.n_parts = (u32)f.pi_K;
      break;
    case CPB_MODEL_PRIMCONN:
      f.net = build_rank(A, RANK_NET);
      f.lcn = build_partwise_rank(A, f.pi_asg.get(), (u32)f.pi_K, f.part_col, f.part_start);
      d.lcn = f.lcn->dev();
      d.part_col = f.part_col.get();
      d.part_start = f.part_start.get();
      d.n_parts = (u32)f.pi_K;
      break;
    default: break;
  }
  if (f.net) d.net = f.net->dev();
  if (f.dianet) d.dianet = f.dianet->dev();
  if (f.selfnet) d.selfnet = f.selfnet->dev();
  if (f.selfpin) d.selfpin = f.selfpin->dev();
  f.ranks_built = true;
}

// ---- oracle_query_batch ---------------------------------------------------------------------------
template <class T>
__global__ void __launch_bounds__(256) k_oracle_query(const __grid_constant__ DevOracle o, i64 Q, const i64* __restrict__ qj,
                                                      const i64* __restrict__ qjp, const i64* __restrict__ qk, double* __restrict__ out) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < (size_t)Q; t += stride) {
    const i64 j = qj[t], jp = qjp[t];
    double r;
    if (j < 1 || jp < j || jp > (i64)o.n + 1) r = __longlong_as_double(0x7ff8000000000000ll);  // invalid query -> NaN
    else if (o.kind == CPB_MODEL_COLBLOCK && jp - j > (i64)o.w_tab) r = __longlong_as_double(0x7ff0000000000000ll);  // wider than the tables: +Inf
    else r = (double)dev_cost<T>(o, (u32)j, (u32)jp, qk ? (u32)qk[t] : 1u);
    out[t] = r;
  }
}

void oracle_query(Oracle& f, i64 Q, const i64* d_j, const i64* d_jp, double* d_cost, const i64* d_k) {
  if (Q <= 0) return;
  if (f.dev.kind == CPB_MODEL_BLOCK) throw Error(CPB_ERR_UNSUPPORTED, "random-access queries of the 2-D block model are served through pack_stripe only");
  oracle_ensure_ranks(f);
  const double L = f.net ? f.net->wm.L : f.dianet ? f.dianet->wm.L : f.selfpin ? f.selfpin->wm.L : 0;
  ProfScope prof("oracle_query_batch", (double)Q * (24.0 + L * 2.0 * 32.0));
  const unsigned grid = (unsigned)std::min<size_t>(((size_t)Q + 255) / 256, (size_t)ctx().sm_count * 16);
  if (f.dev.is_float) CPB_LAUNCH(k_oracle_query<double>, grid, 256, 0, f.dev, Q, d_j, d_jp, d_k, d_cost);
  else CPB_LAUNCH(k_oracle_query<i64>, grid, 256, 0, f.dev, Q, d_j, d_jp, d_k, d_cost);
}

static double query_one(Oracle& f, i64 j, i64 jp) {
  DBuf<i64> q(2);
  DBuf<double> c(1);
  const i64 h[2] = {j, jp};
  CPB_CUDA(cudaMemcpyAsync(q.get(), h, sizeof(h), cudaMemcpyHostToDevice, ctx().stream));
  oracle_query(f, 1, q.get(), q.get() + 1, c.get());
  double r = 0;
  CPB_CUDA(cudaMemcpyAsync(&r, c.get(), sizeof(double), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  return r;
}

// bound_stripe: WorkCosts.jl:37-51, ConnectivityCosts.jl:25-35, Monotonized...:94-105, EnvelopeCosts.jl:44-54
template <class T> static void bound_T(Oracle& f, i64 K, double out[2]) {
  const Matrix& A = *f.A;
  const cpb_model& m = f.mdl;
  T c[5];
  for (int t = 0; t < 5; ++t) c[t] = (T)m.coef[t];
  T c_lo, c_hi;
  switch (m.kind) {
    case CPB_MODEL_WORK: {
      c_lo = c[0] + jl_fld(c[1] * (T)A.n + c[2] * (T)A.N, (T)K);
      if (c[1] >= 0 && c[2] >= 0) c_hi = c[0] + c[1] * (T)A.n + c[2] * (T)A.N;
      else if (c[1] <= 0 && c[2] <= 0) c_hi = c[0];
      else throw Error(CPB_ERR_ARG, "work model coefficients must share a sign (WorkCosts.jl:47)");
      break;
    }
    case CPB_MODEL_CONNECTIVITY: {
      CPB_REQUIRE(c[1] >= 0 && c[2] >= 0 && c[3] >= 0, "negative beta (ConnectivityCosts.jl:29-31)");
      if (f.ranks_built) {
        c_hi = (T)query_one(f, 1, A.n + 1);
      } else {  // ocl(1, n+1) from the link array alone: nets(1, n+1) = number of non-empty rows
        if (!f.ls) f.ls = build_link_stream(*f.A, false, false, false, /*as_pos=*/true);
        if (f.ls->h_first_count < 0) f.ls->h_first_count = count_first_occurrences(*f.ls);
        const i64 nets_all = f.ls->h_first_count;
        c_hi = c[0] + (T)A.n * c[1] + (T)A.N * c[2] + (T)nets_all * c[3];
      }
      c_lo = c[0] + jl_fld(c_hi - c[0], (T)K);
      break;
    }
    case CPB_MODEL_PRIMEDGE: {  // PrimaryEdgeCutCosts.jl:29-40
      CPB_REQUIRE(c[1] >= 0 && c[2] >= 0 && c[3] >= 0, "negative beta (PrimaryEdgeCutCosts.jl:33-35)");
      c_hi = c[0] + c[1] * (T)A.n + std::max(c[2], c[3]) * (T)A.N;
      c_lo = c[0] + jl_fld(c[1] * (T)A.n + std::min(c[2], c[3]) * (T)A.N, (T)K);
      break;
    }
    case CPB_MODEL_SECEDGE: {  // SecondaryEdgeCutCosts.jl:43-60 (oracle form)
      CPB_REQUIRE(c[1] >= 0 && c[2] >= 0 && c[3] >= 0, "negative beta (SecondaryEdgeCutCosts.jl:49-51)");
      oracle_ensure_ranks(f);
      const i64 Kp = f.pi_K;
      std::vector<u32> hs(Kp + 1), hz(Kp);
      CPB_CUDA(cudaMemcpyAsync(hs.data(), f.part_start.get(), (Kp + 1) * sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
      CPB_CUDA(cudaMemcpyAsync(hz.data(), f.pi_size.get(), Kp * sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));
      c_lo = 0; c_hi = 0;
      for (i64 k = 0; k < std::min<i64>(K, Kp); ++k) {
        c_lo = std::max(c_lo, c[0] + (T)(i64)hz[k] * c[1] + (T)(i64)(hs[k + 1] - hs[k]) * std::min(c[2], c[3]));
        c_hi = std::max(c_hi, c[0] + (T)(i64)hz[k] * c[1] + (T)(i64)(hs[k + 1] - hs[k]) * std::max(c[2], c[3]));
      }
      break;
    }
    case CPB_MODEL_SECCONN: {  // SecondaryConnectivityCosts.jl:44-65 (oracle form): maxima over the row parts
      CPB_REQUIRE(c[1] >= 0 && c[2] >= 0 && c[3] >= 0 && c[4] >= 0, "negative beta (SecondaryConnectivityCosts.jl:50-53)");
      oracle_ensure_ranks(f);
      const i64 Kp = f.pi_K;
      std::vector<u32> hs(Kp + 1), hh(Kp + 1), hz(Kp);
      CPB_CUDA(cudaMemcpyAsync(hs.data(), f.part_start.get(), (Kp + 1) * sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
      CPB_CUDA(cudaMemcpyAsync(hz.data(), f.pi_size.get(), Kp * sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));
      for (i64 k = 0; k <= Kp; ++k) CPB_CUDA(cudaMemcpyAsync(&hh[k], f.part_head.get() + hs[k], sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
      CPB_CUDA(cudaStreamSynchronize(ctx().stream));
      c_lo = 0; c_hi = 0;
      for (i64 k = 0; k < std::min<i64>(K, Kp); ++k) {
        const T base = c[0] + (T)(i64)hz[k] * c[1] + (T)(i64)(hs[k + 1] - hs[k]) * c[2];
        c_lo = std::max(c_lo, base);
        c_hi = std::max(c_hi, c[0] + (T)(i64)hz[k] * c[1] + (T)(i64)(hs[k + 1] - hs[k]) * c[2] + (T)(i64)(hh[k + 1] - hh[k]) * c[4]);
      }
      break;
    }
    case CPB_MODEL_PRIMCONN: {  // PrimaryConnectivityCosts.jl:31-42 (oracle form)
      CPB_REQUIRE(c[1] >= 0 && c[2] >= 0 && c[3] >= 0 && c[4] >= 0, "negative beta (PrimaryConnectivityCosts.jl:35-38)");
      oracle_ensure_ranks(f);
      cpb_model conn = f.mdl;  // nets(1, n+1) through a plain connectivity query: (0, 0, 0, 1)
      const DevOracle saved = f.dev;
      f.dev.kind = CPB_MODEL_CONNECTIVITY;
      f.dev.cf[0] = f.dev.cf[1] = f.dev.cf[2] = 0; f.dev.cf[3] = 1;
      f.dev.ci[0] = f.dev.ci[1] = f.dev.ci[2] = 0; f.dev.ci[3] = 1;
      const double nets_all = query_one(f, 1, A.n + 1);
      f.dev = saved;
      (void)conn;
      c_hi = c[0] + c[1] * (T)A.n + c[2] * (T)A.N + std::max(c[3], c[4]) * (T)nets_all;
      c_lo = c[0] + jl_fld(c[1] * (T)A.n + c[2] * (T)A.N, (T)K);
      break;
    }
    case CPB_MODEL_MONOSYM: {
      CPB_REQUIRE(c[1] >= 0 && c[2] >= 0 && c[3] >= 0, "negative beta (Monotonized...:98-100)");
      if (f.h_n_over < 0) {
        u32 n_over = 0;
        CPB_CUDA(cudaMemcpyAsync(&n_over, f.overpos.get() + A.n, sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
        CPB_CUDA(cudaStreamSynchronize(ctx().stream));
        f.h_n_over = n_over;
      }
      const u32 n_over = (u32)f.h_n_over;
      c_hi = c[0] + c[1] * (T)A.n + c[2] * (T)n_over + c[3] * (T)A.m;
      c_lo = c[0] + jl_fld(c_hi - c[0], (T)K);
      break;
    }
    case CPB_MODEL_ENVELOPE: {
      // the oracle form (EnvelopeCosts.jl:30-42), the one partition_stripe(Bisect*) reaches: c_hi = ocl(1, n + 1) with the
      // oracle's own left-to-right sum, c_lo = alpha + fld(c_hi - alpha, K); an empty pattern is fine (envelope width 0)
      CPB_REQUIRE(c[1] >= 0 && c[2] >= 0 && c[3] >= 0, "negative beta (EnvelopeCosts.jl:34-36)");
      c_hi = (T)query_one(f, 1, A.n + 1);
      c_lo = c[0] + jl_fld(c_hi - c[0], (T)K);
      break;
    }
    default: throw Error(CPB_ERR_UNSUPPORTED, "bound_stripe has no method for this model in the reference");
  }
  out[0] = (double)c_lo;
  out[1] = (double)c_hi;
}

void oracle_bound(Oracle& f, i64 K, double out[2]) {
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  if (f.mdl.is_float) bound_T<double>(f, K, out); else bound_T<i64>(f, K, out);
}

double oracle_objective(Oracle& f, bool total, i64 K, const int64_t* h_spl) {
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  std::vector<i64> hj(h_spl, h_spl + K), hjp(h_spl + 1, h_spl + K + 1);
  std::vector<i64> hk(K);
  for (i64 k = 0; k < K; ++k) hk[k] = k + 1;  // part k is charged with the part-k cost (Costs.jl:44-52)
  DBuf<i64> dj(K), djp(K), dk(K);
  DBuf<double> dc(K);
  CPB_CUDA(cudaMemcpyAsync(dj.get(), hj.data(), K * sizeof(i64), cudaMemcpyHostToDevice, ctx().stream));
  CPB_CUDA(cudaMemcpyAsync(djp.get(), hjp.data(), K * sizeof(i64), cudaMemcpyHostToDevice, ctx().stream));
  CPB_CUDA(cudaMemcpyAsync(dk.get(), hk.data(), K * sizeof(i64), cudaMemcpyHostToDevice, ctx().stream));
  oracle_query(f, K, dj.get(), djp.get(), dc.get(), dk.get());
  std::vector<double> hc(K);
  CPB_CUDA(cudaMemcpyAsync(hc.data(), dc.get(), K * sizeof(double), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  double acc = total ? 0.0 : -INFINITY;
  for (i64 k = 0; k < K; ++k) {
    CPB_REQUIRE(!std::isnan(hc[k]), "objective: invalid split vector");
    acc = total ? acc + hc[k] : std::max(acc, hc[k]);
  }
  return acc;
}

// ---- raw color-array queries (netcount & friends) ------------------------------------------------
__global__ void k_count_query(DevRank r, const u32* __restrict__ pos, u32 n, int which, i64 Q, const i64* __restrict__ qj,
                              const i64* __restrict__ qjp, i64* __restrict__ out) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < (size_t)Q; t += stride) {
    const i64 j = qj[t], jp = qjp[t];
    i64 v = -1;
    if (j >= 1 && jp >= j && jp <= (i64)n + 1) {
      if (which == 0) v = (i64)pos[jp - 1] - (i64)pos[j - 1];
      else if (which == RANK_NET || which == RANK_DIANET) v = dev_netcount(r, (u32)j, (u32)jp);
      else v = rank_count_ge(r, (u32)j, (u32)jp);
    }
    out[t] = v;
  }
}

void count_query(Matrix& A, int which, i64 Q, const i64* d_j, const i64* d_jp, i64* d_out) {
  CPB_REQUIRE(which >= 0 && which <= 4, "bad count kind");
  std::unique_ptr<RankStruct> rs;
  DevRank r{};
  if (which != 0) {
    rs = build_rank(A, which);
    r = rs->dev();
  }
  if (Q > 0) CPB_LAUNCH(k_count_query, grid_for((size_t)Q), 256, 0, r, A.pos.get(), (u32)A.n, which, Q, d_j, d_jp, d_out);
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));  // rs is released on return
}

}  // namespace cpb
