// tests/weighted_oracle.cpp -- TEST INFRASTRUCTURE: the CPU oracle's constrained splitters run with a count weight.
//
// ConstrainedCost(f, w, w_max) (Costs.jl:105-147) with w an integer AffineWorkModel, AffineConnectivityModel or
// AffineMonotonizedSymmetricConnectivityModel: the reference turns w into an oracle (oracle_stripe(StepHint(), w, A)) and
// tests w(j, j') > w_max for the windows of every constrained solver.  The restated solvers of oracle/cpo_solvers.hpp reach
// the weight only through `w.over(j, j')`, so they are used here exactly as they are: this file includes them with their
// `Weight` parameter type naming CountWeight below (the oracle's own cpo::Weight holds affine coefficients only).  The
// cost oracles, the weight's oracle and the solvers are all the oracle's restated code; nothing here restates the reference.
#include <chrono>
#include <functional>
#include "../oracle/cpo_core.hpp"

namespace cpo {
// the weight of ConstrainedCost as the weight model's own step oracle
struct CountWeight {
  bool enabled = true;
  i64 w_max = 0;
  std::function<i64(i64, i64)> model;
  inline i64 operator()(i64 j, i64 jp) const { return model(j, jp); }
  inline bool over(i64 j, i64 jp) const { return (*this)(j, jp) > w_max; }
};
}  // namespace cpo

#define Weight CountWeight
#include "../oracle/cpo_solvers.hpp"
#undef Weight

using namespace cpo;

static thread_local std::string g_err;
extern "C" const char* cpw_last_error(void) { return g_err.c_str(); }

static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// oracle/cpo.cpp's with_oracle for the hints the constrained splitters use (step / random)
template <class T, class Fn> static void with_cost_oracle(const cpo_model* mdl, int hint, const Mat& M, const i64* pi_spl, i64 pi_K, Fn fn) {
  if (mdl->kind == CPO_MODEL_BLOCK) throw std::invalid_argument("constrained splitters need a random-access oracle");
  if (mdl->kind == CPO_MODEL_PRIMEDGE || mdl->kind == CPO_MODEL_SECEDGE) {
    if (!pi_spl) throw std::invalid_argument("primary / secondary edge-cut models need a row partition");
    EdgeCutPartOracle<T> f(M, mdl, pi_spl, pi_K, mdl->kind == CPO_MODEL_SECEDGE);
    fn(f);
    return;
  }
  if (mdl->kind == CPO_MODEL_SECCONN) {
    if (!pi_spl) throw std::invalid_argument("secondary connectivity model needs a row partition");
    SecondaryOracle<T> f(M, mdl, pi_spl, pi_K);
    fn(f);
    return;
  }
  auto plain = [&](auto* tag) {
    using Dom = std::remove_pointer_t<decltype(tag)>;
    if (mdl->kind == CPO_MODEL_PRIMCONN) {
      if (!pi_spl) throw std::invalid_argument("primary connectivity model needs a row partition");
      PrimaryOracle<Dom, T> f(M, mdl, pi_spl, pi_K);
      fn(f);
    } else {
      Oracle<Dom, T> f(M, mdl);
      fn(f);
    }
  };
  if (hint == CPO_HINT_STEP) plain((StepDom*)nullptr); else plain((BinDom*)nullptr);
}

// partition_stripe(A, K, method(ConstrainedCost(mdl, wmdl, w_max))) -> spl_out[K+1]; method codes of cpo.h
extern "C" int cpw_partition_stripe_weighted(int method, const cpo_model* mdl, const cpo_model* wmdl, cpo_i64 w_max, const cpo_csc* A,
                                             const cpo_i64* pi_spl, cpo_i64 pi_K, cpo_i64 K, cpo_i64* spl_out, double* seconds_out) {
  try {
    if (K < 1) throw std::invalid_argument("K must be >= 1");
    if (wmdl->is_float) throw std::invalid_argument("weight models take integer coefficients");
    if (wmdl->kind != CPO_MODEL_WORK && wmdl->kind != CPO_MODEL_CONNECTIVITY && wmdl->kind != CPO_MODEL_MONOSYM)
      throw std::invalid_argument("weight must be an AffineWorkModel, AffineConnectivityModel or AffineMonotonizedSymmetricConnectivityModel");
    const int nb = wmdl->kind == CPO_MODEL_WORK ? 2 : 3;
    for (int t = 1; t <= nb; ++t)
      if (wmdl->coef[t] < 0) throw std::invalid_argument("weight models need non-negative betas (monotone windows)");
    Mat M(A);
    const i64 n = M.n;
    ivec spl(K + 2, 0);
    double t0 = now_s(), t1 = t0;
    Oracle<StepDom, i64> wo(M, wmdl);  // oracle_stripe(StepHint(), w, A)
    CountWeight w;
    w.w_max = w_max;
    w.model = [&wo](i64 j, i64 jp) { return wo(j, jp); };
    auto run = [&](auto* tt) {
      using T = std::remove_pointer_t<decltype(tt)>;
      switch (method) {
        case CPO_SPLIT_DYNAMIC_BOTTLENECK: case CPO_SPLIT_DYNAMIC_TOTAL:
          with_cost_oracle<T>(mdl, CPO_HINT_STEP, M, pi_spl, pi_K, [&](auto& f) {
            t1 = now_s();
            using F = std::remove_reference_t<decltype(f)>;
            dynamic_splitter_constrained<F, T>(f, w, n, K, method == CPO_SPLIT_DYNAMIC_TOTAL, spl.data());
          });
          break;
        case CPO_SPLIT_DYNAMIC_BOTTLENECK_CHUNKER: case CPO_SPLIT_DYNAMIC_TOTAL_CHUNKER:
          if (mdl->kind >= CPO_MODEL_PRIMCONN && mdl->kind <= CPO_MODEL_SECEDGE)
            throw std::invalid_argument("chunker-form K-DP on a row-partition-aware model (no method f(j, j') without k in the reference)");
          with_cost_oracle<T>(mdl, CPO_HINT_STEP, M, pi_spl, pi_K, [&](auto& f) {
            t1 = now_s();
            using F = std::remove_reference_t<decltype(f)>;
            dynamic_chunker_kform_constrained<F, T>(f, w, n, K, method == CPO_SPLIT_DYNAMIC_TOTAL_CHUNKER, spl.data());
          });
          break;
        case CPO_SPLIT_CONVEX_TOTAL: case CPO_SPLIT_CONCAVE_TOTAL:
          with_cost_oracle<T>(mdl, CPO_HINT_RANDOM, M, pi_spl, pi_K, [&](auto& f) {
            t1 = now_s();
            using F = std::remove_reference_t<decltype(f)>;
            convex_total_splitter_constrained<F, T>(f, w, n, K, spl.data(), method == CPO_SPLIT_CONCAVE_TOTAL);
          });
          break;
        default: throw std::invalid_argument("weighted constraints are taken by the Dynamic, Convex and Concave total splitters only");
      }
    };
    if (mdl->is_float) run((double*)nullptr); else run((i64*)nullptr);
    const double t2 = now_s();
    for (i64 k = 1; k <= K + 1; ++k) spl_out[k - 1] = spl[k];
    if (seconds_out) { seconds_out[0] = t1 - t0; seconds_out[1] = t2 - t1; }
  } catch (const std::exception& e) {
    g_err = e.what();
    return -1;
  } catch (...) {
    g_err = "unknown error";
    return -1;
  }
  return 0;
}
