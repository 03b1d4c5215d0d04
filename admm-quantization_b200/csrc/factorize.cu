// factorize.cu - the whole outer AO-ADMM loop behind one C-ABI call (admmq_factorize_cp3 / admmq_factorize_mat).
// Replaces the loop of scripts/factorize.py:207-266 (3-D) and :269-310 (2-D): per sweep and mode the Gram-Hadamard
// product, the MTTKRP, the ridge-system inverse, the persistent ADMM kernel and the re-projection, then the two
// reconstruction errors and the reference's stop rules (:259-263 / :303-307).  Host orchestration only: every kernel is
// one of the library's own entry points, enqueued on the caller's stream; the call synchronises once per sweep to read
// the two error sums and the loop reports (the reference synchronises there as well, through `.item()`).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>
#include "common.cuh"

namespace admmq {

struct Carve {
  size_t off = 0;
  size_t take(size_t bytes) {
    const size_t o = off;
    off += align_up(std::max<size_t>(bytes, 16), 256);
    return o;
  }
};

struct FactorizeLayout {
  size_t unf[3], perm[3], G, F, Minv, Minv64, scalars, reports, err, ws_inv, ws_loop, ws_proj, ws_mttkrp, ws_err, total;
  size_t n_inv, n_loop, n_proj, n_mttkrp, n_err;
  int nx[3], ny[3];
};

static FactorizeLayout factorize_layout(int ndim, const int* shape, int R, const admmq_factorize_params* p) {
  FactorizeLayout l;
  memset(&l, 0, sizeof(l));
  Carve c;
  size_t numel = 1;
  int maxd = 0;
  for (int m = 0; m < ndim; ++m) {
    numel *= (size_t)shape[m];
    maxd = std::max(maxd, shape[m]);
  }
  for (int m = 0; m < ndim; ++m) {
    int o0 = -1, o1 = -1;
    for (int k = 0; k < ndim; ++k)
      if (k != m) (o0 < 0 ? o0 : o1) = k;
    l.nx[m] = shape[o0];
    l.ny[m] = (ndim == 3) ? shape[o1] : 1;
  }
  for (int m = 1; m < ndim; ++m) l.unf[m] = c.take(numel * sizeof(float));  // mode 0 is W itself
  if (p->mttkrp_precision == 1)
    for (int m = 0; m < ndim; ++m) l.perm[m] = c.take((size_t)shape[m] * l.ny[m] * ((l.nx[m] + 3) / 4 * 4) * sizeof(float));
  l.G = c.take((size_t)R * R * sizeof(float));
  l.F = c.take((size_t)maxd * R * sizeof(float));
  l.Minv = c.take((size_t)R * admmq_padded_ld(R) * sizeof(float));
  l.Minv64 = c.take(p->solve_precision == 0 ? (size_t)R * admmq_padded_ld(R) * sizeof(double) : 0);
  l.scalars = c.take(64);
  l.reports = c.take(3 * sizeof(admmq_loop_report));
  l.err = c.take(4 * sizeof(double));
  for (int m = 0; m < ndim; ++m) {
    l.n_loop = std::max(l.n_loop, admmq_admm_loop_workspace_bytes(shape[m], R, p->num_attempts));
    l.n_mttkrp = std::max(l.n_mttkrp, p->mttkrp_precision == 1 ? admmq_mttkrp_tc_workspace_bytes(shape[m], l.nx[m], l.ny[m], R)
                                                                : admmq_mttkrp_workspace_bytes(shape[m], l.nx[m], l.ny[m], R, 0));
  }
  l.n_inv = admmq_spd_inverse_workspace_bytes(R);
  l.n_proj = admmq_project_workspace_bytes((int64_t)maxd * R, p->num_attempts);
  l.n_err = admmq_recon_error_workspace_bytes(shape[0], l.nx[0], l.ny[0]);
  l.ws_inv = c.take(l.n_inv);
  l.ws_loop = c.take(l.n_loop);
  l.ws_proj = c.take(l.n_proj);
  l.ws_mttkrp = c.take(l.n_mttkrp);
  l.ws_err = c.take(l.n_err);
  l.total = c.off;
  return l;
}

static int check_params(const char* who, int ndim, const int* shape, int R, const admmq_factorize_params* p) {
  if (p == nullptr || shape == nullptr) return fail(ADMMQ_E_BADARG, "%s: null argument", who);
  if (ndim != 2 && ndim != 3) return fail(ADMMQ_E_BADARG, "%s: Incorrect number of dimentions in weight tensor (%d)", who, ndim);
  for (int m = 0; m < ndim; ++m)
    if (shape[m] <= 0) return fail(ADMMQ_E_BADARG, "%s: empty mode %d", who, m);
  if (R <= 0) return fail(ADMMQ_E_BADARG, "%s: rank must be positive", who);
  if (p->max_iter_als < 1 || p->max_iter_admm < 1) return fail(ADMMQ_E_BADARG, "%s: iteration budgets must be >= 1", who);
  if (p->bits < 1 || p->bits > 8) return fail(ADMMQ_E_BADARG, "%s: bits must be in 1..8", who);
  if (!known_scheme(p->qscheme)) return fail(ADMMQ_E_BADARG, "%s: unknown qscheme %d", who, p->qscheme);
  if (int e = check_scheme_bits(who, p->qscheme, p->bits)) return e;
  if (p->solve_precision < 0 || p->solve_precision > 2 || p->mttkrp_precision < 0 || p->mttkrp_precision > 1)
    return fail(ADMMQ_E_BADARG, "%s: solve_precision must be 0..2, mttkrp_precision 0 or 1", who);
  return ADMMQ_OK;
}

static float finish_error(const double* sums) {  // source/admm.py:15 in float32
  const float num = (float)sums[0], den = (float)sums[1];
  return sqrtf(num / den);
}

// One layer's run: set-up once, then enqueue_sweep() / collect() per outer iteration, so that several runs can be
// interleaved on their own streams (admmq_factorize_batch).
struct Run {
  const float* W = nullptr;
  int ndim = 0, shape[3] = {0, 0, 0}, R = 0;
  float* factors[3] = {nullptr, nullptr, nullptr};
  float* duals[3] = {nullptr, nullptr, nullptr};
  float* factors_q[3] = {nullptr, nullptr, nullptr};
  admmq_factorize_params prm;
  float* loss_hist = nullptr;
  float* loss_quant_hist = nullptr;
  int* sweeps_done = nullptr;
  char* ws = nullptr;
  cudaStream_t stream = nullptr;
  FactorizeLayout l;
  const float* unf[3] = {nullptr, nullptr, nullptr};
  std::vector<float> hist;
  int n_hist = 0, sweep = 0;
  bool active = true;

  int errors_of(float* const* fac, double* out) {
    return admmq_recon_error(W, shape[0], fac[0], fac[1], l.nx[0], ndim == 3 ? fac[2] : nullptr, l.ny[0], R, out,
                             ws + l.ws_err, l.n_err, (void*)stream);
  }
  float* G() { return (float*)(ws + l.G); }
  float* F() { return (float*)(ws + l.F); }
  float* Minv() { return (float*)(ws + l.Minv); }
  double* Minv64() { return prm.solve_precision == 0 ? (double*)(ws + l.Minv64) : nullptr; }
  float* rho() { return (float*)(ws + l.scalars); }
  int* inv_status() { return (int*)(ws + l.scalars + 16); }
  admmq_loop_report* reports() { return (admmq_loop_report*)(ws + l.reports); }
  double* err() { return (double*)(ws + l.err); }

  int init(const float* W_, int ndim_, const int* shape_, int R_, float* const* fac, float* const* du, float* const* fq,
           const admmq_factorize_params* p, float* lh, float* lqh, int* done, void* workspace, size_t workspace_bytes,
           cudaStream_t stream_) {
    if (int e = check_params("admmq_factorize", ndim_, shape_, R_, p)) return e;
    if (W_ == nullptr || fac == nullptr || du == nullptr || fq == nullptr || lh == nullptr || lqh == nullptr || done == nullptr)
      return fail(ADMMQ_E_BADARG, "admmq_factorize: null pointer");
    for (int m = 0; m < ndim_; ++m)
      if (fac[m] == nullptr || du[m] == nullptr || fq[m] == nullptr)
        return fail(ADMMQ_E_BADARG, "admmq_factorize: null factor pointer for mode %d", m);
    W = W_;
    ndim = ndim_;
    R = R_;
    prm = *p;
    for (int m = 0; m < ndim; ++m) {
      shape[m] = shape_[m];
      factors[m] = fac[m];
      duals[m] = du[m];
      factors_q[m] = fq[m];
    }
    loss_hist = lh;
    loss_quant_hist = lqh;
    sweeps_done = done;
    stream = stream_;
    l = factorize_layout(ndim, shape, R, &prm);
    if (workspace == nullptr || workspace_bytes < l.total || ((uintptr_t)workspace & 255) != 0)
      return fail(ADMMQ_E_WORKSPACE, "admmq_factorize: workspace needs %zu bytes, 256-byte aligned", l.total);
    ws = (char*)workspace;
    void* st = (void*)stream;
    *sweeps_done = 0;
    // ---- once per run: unfoldings (and their (m, y, x) permutations for the tensor-core MTTKRP)
    unf[0] = W;
    if (ndim == 3) {
      for (int m = 1; m < 3; ++m) {
        if (int e = admmq_unfold3(W, shape[0], shape[1], shape[2], m, (float*)(ws + l.unf[m]), st)) return e;
        unf[m] = (const float*)(ws + l.unf[m]);
      }
    } else {
      // W^T as the mode-1 unfolding of the I x J x 1 tensor
      if (int e = admmq_unfold3(W, shape[0], shape[1], 1, 1, (float*)(ws + l.unf[1]), st)) return e;
      unf[1] = (const float*)(ws + l.unf[1]);
    }
    if (prm.mttkrp_precision == 1)
      for (int m = 0; m < ndim; ++m)
        if (int e = admmq_permute_myx(unf[m], shape[m], l.nx[m], l.ny[m], (float*)(ws + l.perm[m]), st)) return e;
    if (!prm.init_is_random) {  // scripts/factorize.py:192-201: errors of the initial factors and of their projection
      for (int m = 0; m < ndim; ++m)
        if (int e = admmq_project(factors[m], (int64_t)shape[m] * R, prm.bits, prm.qscheme, prm.num_attempts, nullptr,
                                  nullptr, factors_q[m], nullptr, nullptr, ws + l.ws_proj, l.n_proj, st))
          return e;
      if (int e = errors_of(factors, err())) return e;
      if (int e = errors_of(factors_q, err() + 2)) return e;
      double h[4];
      ADMMQ_CUDA_OK(cudaMemcpyAsync(h, err(), sizeof(h), cudaMemcpyDeviceToHost, stream));
      ADMMQ_CUDA_OK(cudaStreamSynchronize(stream));
      loss_hist[n_hist] = finish_error(h);
      loss_quant_hist[n_hist] = finish_error(h + 2);
      hist.push_back(loss_hist[n_hist]);
      ++n_hist;
    }
    active = sweep < prm.max_iter_als;
    return ADMMQ_OK;
  }

  // one outer iteration on the run's stream, no host synchronisation (scripts/factorize.py:214-255)
  int enqueue_sweep() {
    void* st = (void*)stream;
    for (int m = 0; m < ndim; ++m) {
      int o0 = -1, o1 = -1;
      for (int k = 0; k < ndim; ++k)
        if (k != m) (o0 < 0 ? o0 : o1) = k;
      const float* X = factors[o0];
      const float* Y = ndim == 3 ? factors[o1] : nullptr;
      if (int e = admmq_gram_hadamard(X, l.nx[m], Y, Y ? l.ny[m] : 0, R, G(), st)) return e;                    // :215
      if (prm.mttkrp_precision == 1) {
        if (int e = admmq_mttkrp_tc((const float*)(ws + l.perm[m]), shape[m], X, l.nx[m], Y, l.ny[m], R, F(),
                                    ws + l.ws_mttkrp, l.n_mttkrp, st))
          return e;
      } else if (int e = admmq_mttkrp(unf[m], shape[m], X, l.nx[m], Y, l.ny[m], R, F(), 0, ws + l.ws_mttkrp, l.n_mttkrp, st)) {
        return e;                                                                                              // :217
      }
      if (int e = admmq_spd_inverse(G(), R, Minv(), Minv64(), rho(), inv_status(), prm.max_ctas, ws + l.ws_inv, l.n_inv, st)) return e;
      if (int e = admmq_admm_loop(factors[m], duals[m], F(), Minv(), Minv64(), rho(), inv_status(), shape[m], R, prm.max_iter_admm,
                                  prm.eps, prm.bits, prm.qscheme, prm.num_attempts, prm.solve_precision, prm.max_ctas,
                                  nullptr, reports() + m, ws + l.ws_loop, l.n_loop, st))
        return e;                                                                                              // :218
      if (int e = admmq_project(factors[m], (int64_t)shape[m] * R, prm.bits, prm.qscheme, prm.num_attempts, nullptr, nullptr,
                                factors_q[m], nullptr, nullptr, ws + l.ws_proj, l.n_proj, st))
        return e;                                                                                              // :222
    }
    if (int e = errors_of(factors, err())) return e;        // :246-248
    if (int e = errors_of(factors_q, err() + 2)) return e;  // :249-253
    return ADMMQ_OK;
  }

  // host side of the sweep: synchronise the stream, append the errors, apply the stop rules (:259-263 / :303-307)
  int collect() {
    double h[4];
    admmq_loop_report rep[3];
    ADMMQ_CUDA_OK(cudaMemcpyAsync(h, err(), sizeof(h), cudaMemcpyDeviceToHost, stream));
    ADMMQ_CUDA_OK(cudaMemcpyAsync(rep, reports(), (size_t)ndim * sizeof(admmq_loop_report), cudaMemcpyDeviceToHost, stream));
    ADMMQ_CUDA_OK(cudaStreamSynchronize(stream));
    for (int m = 0; m < ndim; ++m)
      if (rep[m].status == ADMMQ_E_NOT_PD)
        return fail(ADMMQ_E_NOT_PD, "admmq_factorize: G + rho*I is not positive-definite (mode %d, sweep %d)", m, sweep);
    loss_hist[n_hist] = finish_error(h);
    loss_quant_hist[n_hist] = finish_error(h + 2);
    hist.push_back(loss_hist[n_hist]);
    ++n_hist;
    ++sweep;
    *sweeps_done = sweep;
    const size_t n = hist.size();
    if (n > 1 && std::fabs((double)hist[n - 2] - (double)hist[n - 1]) < prm.tol) active = false;
    const size_t back = ndim == 3 ? 5 : 10;
    if (n > 10 && (double)hist[n - 1] - (double)hist[n - back] > 1e-3) active = false;
    if (sweep >= prm.max_iter_als) active = false;
    return ADMMQ_OK;
  }
};

static int factorize(const float* W, int ndim, const int* shape, int R, float* const* factors, float* const* duals,
                     float* const* factors_q, const admmq_factorize_params* p, float* loss_hist, float* loss_quant_hist,
                     int* sweeps_done, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  Run run;
  if (int e = run.init(W, ndim, shape, R, factors, duals, factors_q, p, loss_hist, loss_quant_hist, sweeps_done, workspace,
                       workspace_bytes, stream))
    return e;
  while (run.active) {
    if (int e = run.enqueue_sweep()) return e;
    if (int e = run.collect()) return e;
  }
  return ADMMQ_OK;
}

}  // namespace admmq

using namespace admmq;

extern "C" size_t admmq_factorize_workspace_bytes(int ndim, const int* shape, int R, const admmq_factorize_params* params) {
  if (check_params("admmq_factorize_workspace_bytes", ndim, shape, R, params)) return 0;
  return factorize_layout(ndim, shape, R, params).total;
}

extern "C" int admmq_factorize_cp3(const float* W, int I, int J, int K, int R, float* A, float* B, float* C, float* UA,
                                   float* UB, float* UC, float* Aq, float* Bq, float* Cq,
                                   const admmq_factorize_params* params, float* loss_hist, float* loss_quant_hist,
                                   int* sweeps_done, void* workspace, size_t workspace_bytes, void* stream) {
  const int shape[3] = {I, J, K};
  float* fac[3] = {A, B, C};
  float* du[3] = {UA, UB, UC};
  float* fq[3] = {Aq, Bq, Cq};
  return factorize(W, 3, shape, R, fac, du, fq, params, loss_hist, loss_quant_hist, sweeps_done, workspace, workspace_bytes,
                   (cudaStream_t)stream);
}

extern "C" int admmq_factorize_mat(const float* W, int I, int J, int R, float* A, float* B, float* UA, float* UB, float* Aq,
                                   float* Bq, const admmq_factorize_params* params, float* loss_hist,
                                   float* loss_quant_hist, int* sweeps_done, void* workspace, size_t workspace_bytes,
                                   void* stream) {
  const int shape[2] = {I, J};
  float* fac[2] = {A, B};
  float* du[2] = {UA, UB};
  float* fq[2] = {Aq, Bq};
  return factorize(W, 2, shape, R, fac, du, fq, params, loss_hist, loss_quant_hist, sweeps_done, workspace, workspace_bytes,
                   (cudaStream_t)stream);
}

// Independent solves side by side (BASELINE configs 2, 3, 5: layers x reduction rates x bit-widths): every problem
// is enqueued on ITS OWN stream with its own cooperative-grid budget (params.max_ctas), sweep by sweep, and the host
// collects the errors of all active problems after each round, so the solves overlap on the GPU like the streams of
// scripts/factorize_model.py.  A problem that stops (stop rules or budget) simply drops out of the rounds.
extern "C" int admmq_factorize_batch(int n_problems, const admmq_problem* problems) {
  if (n_problems <= 0 || problems == nullptr) return fail(ADMMQ_E_BADARG, "admmq_factorize_batch: no problems");
  std::vector<Run> runs((size_t)n_problems);
  for (int k = 0; k < n_problems; ++k) {
    const admmq_problem& q = problems[k];
    if (int e = runs[k].init(q.W, q.ndim, q.shape, q.rank, q.factors, q.duals, q.factors_q, &q.params, q.loss_hist,
                             q.loss_quant_hist, q.sweeps_done, q.workspace, q.workspace_bytes, (cudaStream_t)q.stream))
      return e;
  }
  for (;;) {
    bool any = false;
    for (auto& r : runs)
      if (r.active) {
        any = true;
        if (int e = r.enqueue_sweep()) return e;
      }
    if (!any) break;
    for (auto& r : runs)
      if (r.active)
        if (int e = r.collect()) return e;
  }
  return ADMMQ_OK;
}
