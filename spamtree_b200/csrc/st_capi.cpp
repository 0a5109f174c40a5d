// st_capi.cpp — the extern "C" boundary declared in include/spamtree_b200.h.  No exception leaves this file.
#include <cmath>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/spamtree_b200.h"
#include "st_kernels.cuh"
#include <cuda_runtime.h>

#include "st_mh.hpp"
#include "st_model.hpp"
#include "st_tree.hpp"

namespace st {
int mcmc_run(Model& M, const st_mcmc_opts& o, st_mcmc_out& out);
}

struct st_handle {
  st::Model model;
};
struct st_tree {
  st::TreeResult t;
};

static thread_local std::string g_create_error;

#define ST_GUARD_BEGIN try {
#define ST_GUARD_END(h)                                                   \
  }                                                                       \
  catch (const std::bad_alloc&) {                                         \
    if (h) (h)->model.err = "out of host memory";                         \
    return ST_ERR_INVALID;                                                \
  }                                                                       \
  catch (const std::exception& ex) {                                      \
    if (h) (h)->model.err = ex.what();                                    \
    return ST_ERR_INVALID;                                                \
  }                                                                       \
  catch (...) {                                                           \
    if (h) (h)->model.err = "unknown exception";                          \
    return ST_ERR_INVALID;                                                \
  }

static void csr_assign(st::CSR& c, const int64_t* ptr, const int64_t* idx, int64_t n) {
  c.ptr.assign(ptr, ptr + n + 1);
  c.idx.assign(idx, idx + ptr[n]);
}

// every entry point that touches device state makes the handle's GPU the calling thread's current device first (a host may
// hold handles on several GPUs; streams, launches and the shared-memory opt-in are all per device)
static inline void activate(st_handle* h) {
  if (h && h->model.device >= 0) cudaSetDevice(h->model.device);
}

extern "C" {

const char* st_version(void) { return "spamtree_b200 0.1 sm_100a"; }

int st_create(const st_problem* pr, st_handle** out) {
  if (!pr || !out) return ST_ERR_INVALID;
  *out = nullptr;
  st_handle* h = nullptr;
  try {
    if (pr->n_all <= 0 || pr->p <= 0 || pr->q <= 0 || pr->n_blocks <= 0) { g_create_error = "empty problem"; return ST_ERR_INVALID; }
    h = new st_handle();
    st::Model& M = h->model;
    M.n_all = pr->n_all; M.p = pr->p; M.q = pr->q; M.n_blocks = pr->n_blocks;
    M.y.assign(pr->y, pr->y + pr->n_all);
    M.X.assign(pr->X, pr->X + (size_t)pr->n_all * pr->p);
    M.coords.assign(pr->coords, pr->coords + (size_t)pr->n_all * 2);
    M.mv_id.assign(pr->mv_id, pr->mv_id + pr->n_all);
    csr_assign(M.indexing, pr->indexing_ptr, pr->indexing_idx, pr->n_blocks);
    csr_assign(M.parents, pr->parents_ptr, pr->parents_idx, pr->n_blocks);
    csr_assign(M.children, pr->children_ptr, pr->children_idx, pr->n_blocks);
    M.block_names.assign(pr->block_names, pr->block_names + pr->n_blocks);
    M.block_groups.assign(pr->block_groups, pr->block_groups + pr->n_blocks);
    M.res_is_ref.assign(pr->res_is_ref, pr->res_is_ref + pr->n_res);
    M.keep_H = pr->keep_H != 0;
    M.limited = pr->limited_tree != 0;
    M.device = pr->device;
    if (pr->smem_panel_bytes > 0) M.smem_budget = (size_t)pr->smem_panel_bytes;
    M.theta[0].assign(pr->theta, pr->theta + pr->n_theta);
    M.theta[1] = M.theta[0];
    M.Bcoeff.assign((size_t)pr->p * pr->q, 0.0);
    for (int j = 0; j < pr->q; j++)
      for (int a = 0; a < pr->p; a++) M.Bcoeff[a + (size_t)j * pr->p] = pr->beta[a];  // spamtree_model.cpp:124-129
    M.tausq_inv.assign(pr->q, 1.0 / pr->tausq);                                         // :118
    M.rng.seed(1);
    if (pr->partition && pr->partition->nranks > 1) {
      const st_partition& pt = *pr->partition;
      if (pt.rank < 0 || pt.rank >= pt.nranks) { g_create_error = "partition: bad rank"; delete h; return ST_ERR_INVALID; }
      M.part = true;
      M.rank = pt.rank; M.nranks = pt.nranks; M.n_top_levels = pt.n_top_levels;
      M.rng_row_offset = pt.rng_row_offset; M.n_global_rows = pt.n_global_rows;
      // every random stream is keyed by the row's id in the whole problem (device) or drawn for all of its rows (host): without
      // the map the ranks would draw different numbers for the rows they share
      if (!pt.global_rows || pt.n_global_rows < pr->n_all) { g_create_error = "partition: global_rows / n_global_rows missing"; delete h; return ST_ERR_INVALID; }
      for (int64_t i = 0; i < pr->n_all; i++)
        if (pt.global_rows[i] < 0 || pt.global_rows[i] >= pt.n_global_rows) { g_create_error = "partition: global row out of range"; delete h; return ST_ERR_INVALID; }
      M.global_rows.assign(pt.global_rows, pt.global_rows + pr->n_all);
      M.allreduce_fn = pt.allreduce; M.allreduce_ctx = pt.ctx;
    }
    {
      st::CovTab tab;
      std::string e;
      if (!st::make_covtab(M.theta[0].data(), pr->n_theta, pr->q, tab, e)) { g_create_error = e; delete h; return ST_ERR_INVALID; }
    }
    std::string e;
    int rc = M.init(e);
    if (rc) { g_create_error = e.empty() ? M.err : e; delete h; return rc; }
    *out = h;
    return ST_OK;
  } catch (const std::exception& ex) {
    g_create_error = ex.what();
  } catch (...) {
    g_create_error = "unknown exception";
  }
  delete h;
  return ST_ERR_INVALID;
}

void st_destroy(st_handle* h) {
  activate(h);
  delete h;
}

const char* st_last_error(const st_handle* h) { return h ? h->model.err.c_str() : g_create_error.c_str(); }

int st_theta_update(st_handle* h, int slot, const double* theta) {
  if (!h || !theta) return ST_ERR_INVALID;
  ST_GUARD_BEGIN return h->model.theta_update(slot, theta);
  ST_GUARD_END(h)
}
int st_get_loglik_comps_w(st_handle* h, int slot, double* out3) {
  if (!h || !out3) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.get_loglik_comps_w(slot, out3);
  ST_GUARD_END(h)
}
int st_deal_with_w(st_handle* h, const double* z, uint64_t seed) {
  if (!h) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.deal_with_w(z, seed);
  ST_GUARD_END(h)
}
int st_get_loglik_w(st_handle* h, int slot, double* out2) {
  if (!h || !out2) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.get_loglik_w(slot, out2);
  ST_GUARD_END(h)
}
int st_accept_make_change(st_handle* h) {
  if (!h) return ST_ERR_INVALID;
  if (h->model.alter_scratch) {
    h->model.err = "the alter slot holds a BUILD of st_predict_new: st_get_loglik_comps_w(h, 1, ...) rebuilds it first";
    return ST_ERR_INVALID;
  }
  activate(h);
  h->model.accept_make_change();
  return ST_OK;
}
int st_predict(st_handle* h, int theta_changed) {
  if (!h) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.predict(theta_changed != 0);
  ST_GUARD_END(h)
}
int st_gibbs_sample_beta(st_handle* h, const double* zb, int faithful_index) {
  if (!h) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.gibbs_sample_beta(zb, faithful_index != 0);
  ST_GUARD_END(h)
}
int st_gibbs_sample_tausq(st_handle* h, const double* fixed) {
  if (!h) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.gibbs_sample_tausq(fixed);
  ST_GUARD_END(h)
}
int st_seed(st_handle* h, uint64_t seed) {
  if (!h) return ST_ERR_INVALID;
  h->model.rng.seed(seed);
  return ST_OK;
}
int st_get_w(st_handle* h, double* w_out) {
  if (!h || !w_out) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.get_w(w_out);
  ST_GUARD_END(h)
}
int st_set_w(st_handle* h, const double* w_in) {
  if (!h || !w_in) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.set_w(w_in);
  ST_GUARD_END(h)
}
int st_get_params(st_handle* h, double* Bcoeff, double* tausq_inv, double* XB) {
  if (!h) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN
  st::Model& M = h->model;
  if (Bcoeff) std::copy(M.Bcoeff.begin(), M.Bcoeff.end(), Bcoeff);
  if (tausq_inv) std::copy(M.tausq_inv.begin(), M.tausq_inv.end(), tausq_inv);
  if (XB) return M.get_xb(XB);
  return ST_OK;
  ST_GUARD_END(h)
}
int st_set_tausq_inv(st_handle* h, const double* t) {
  if (!h || !t) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.set_tausq_inv(t);
  ST_GUARD_END(h)
}
int st_get_node_state(st_handle* h, int slot, int u, const char* which, double* out, int64_t cap, int64_t* count) {
  if (!h || !which || !count) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.get_node_state(slot, u, which, out, cap, count);
  ST_GUARD_END(h)
}
int st_get_index(st_handle* h, const char* which, int u, int c, int64_t* out, int64_t cap, int64_t* count) {
  if (!h || !which || !count) return ST_ERR_INVALID;
  ST_GUARD_BEGIN return h->model.get_index(which, u, c, out, cap, count);
  ST_GUARD_END(h)
}
int st_mcmc_run(st_handle* h, const st_mcmc_opts* opts, st_mcmc_out* out) {
  if (!h || !opts || !out || !opts->set_unif_bounds || !opts->mcmcsd || opts->keep < 0 || opts->thin < 1) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return st::mcmc_run(h->model, *opts, *out);
  ST_GUARD_END(h)
}
int st_predict_new(st_handle* h, const st_new_rows* rows, const st_pred_samples* samples, st_pred_out* out) {
  if (!h || !rows || !samples || !out) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.predict_new(*rows, *samples, *out);
  ST_GUARD_END(h)
}
int st_keep_samples_on_device(st_handle* h, int32_t what) {
  if (!h) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.keep_samples_on_device(what);
  ST_GUARD_END(h)
}
int st_get_loglik_int(st_handle* h, double* out) {
  if (!h || !out) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.get_loglik_int(out);
  ST_GUARD_END(h)
}
int st_copy_store(st_handle* h, int32_t which, double* out, int64_t* n_rows, int32_t* n_samples) {
  if (!h) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.copy_store(which, out, n_rows, n_samples);
  ST_GUARD_END(h)
}
int st_summarize(st_handle* h, int32_t which, const double* probs, int32_t n_probs, st_summary_out* out) {
  if (!h || !out) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.summarize(which, probs, n_probs, *out);
  ST_GUARD_END(h)
}
int st_predict_new_stored(st_handle* h, const st_new_rows* rows, uint64_t seed, int32_t keep_draws, st_pred_out* out) {
  if (!h || !rows || !out) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN
  st_pred_samples ps{};
  ps.seed = seed;
  return h->model.predict_new(*rows, ps, *out, true, keep_draws != 0);
  ST_GUARD_END(h)
}
int st_summarize_chains(st_handle* const* hs, int32_t n_chains, int32_t which, const double* probs, int32_t n_probs,
                        st_chains_summary_out* out) {
  if (!hs || n_chains < 1 || !hs[0]) {  // (no handle to report to)
    g_create_error = n_chains < 1 ? "st_summarize_chains: n_chains must be at least 1" : "st_summarize_chains: hs or hs[0] is NULL";
    return ST_ERR_INVALID;
  }
  st_handle* h0 = hs[0];
  st::Model& M0 = h0->model;
  if (!out) { M0.err = "st_summarize_chains: out is NULL"; return ST_ERR_INVALID; }
  activate(h0);
  ST_GUARD_BEGIN
  if (which < 0 || which > 3) { M0.err = "st_summarize_chains: which must be 0 (w), 1 (yhat), 2 (w_new) or 3 (y_new)"; return ST_ERR_INVALID; }
  const int64_t n = M0.store.get(which).n;
  const int S = M0.store.get(which).S;
  int rc = st::chains_check("st_summarize_chains", n_chains, std::max(S, 1), probs, n_probs, M0.err);
  if (rc) return rc;
  std::vector<const double*> src(n_chains);
  for (int k = 0; k < n_chains; k++) {
    const std::string hk = "st_summarize_chains: handle " + std::to_string(k);
    if (!hs[k]) { M0.err = hk + " is NULL"; return ST_ERR_INVALID; }
    const st::Model& Mk = hs[k]->model;
    if (Mk.device != M0.device) {
      M0.err = hk + " is on device " + std::to_string(Mk.device) + ", handle 0 on device " + std::to_string(M0.device);
      return ST_ERR_INVALID;
    }
    const st::DrawStore::Store* s = Mk.store.find(which, hk + " has ", M0.err);
    if (!s) return ST_ERR_INVALID;
    if (s->n != n || s->S != S) {
      M0.err = hk + " stores " + std::to_string(s->S) + " draws of " + std::to_string(s->n) + " rows, handle 0 " + std::to_string(S) +
               " draws of " + std::to_string(n) + " rows";
      return ST_ERR_INVALID;
    }
    src[k] = s->d;
  }
  for (int k = 1; k < n_chains; k++)  // every store is complete before the kernel reads it on hs[0]'s stream
    if (const cudaError_t e = cudaStreamSynchronize(hs[k]->model.stream)) {
      M0.err = std::string("st_summarize_chains: CUDA error in sync of handle ") + std::to_string(k) + ": " + cudaGetErrorString(e);
      return ST_ERR_CUDA;
    }
  return st::summarize_chains(src.data(), n, n_chains, S, probs, n_probs, *out, M0.stream, M0.err);
  ST_GUARD_END(h0)
}
int st_summarize_draws(int32_t device, const double* draws, int64_t n_rows, int32_t n_chains, int32_t n_samples,
                       const double* probs, int32_t n_probs, st_chains_summary_out* out) {
  if (!out || n_rows < 0 || (n_rows > 0 && !draws)) { g_create_error = "st_summarize_draws: out or draws missing, or n_rows < 0"; return ST_ERR_INVALID; }
  try {
    int rc = st::chains_check("st_summarize_draws", n_chains, n_samples, probs, n_probs, g_create_error);
    if (rc) return rc;
    const size_t all = (size_t)n_rows * n_samples * n_chains;
    for (size_t j = 0; j < all; j++)
      if (!std::isfinite(draws[j])) {
        g_create_error = "st_summarize_draws: draw " + std::to_string(j) + " ([chain][sample][row] order) is not finite";
        return ST_ERR_INVALID;
      }
    const bool any = out->mean || out->sd || out->quantiles || out->rhat || out->ess_bulk || out->ess_tail;
    if (!any || n_rows == 0) return st::summarize_chains(nullptr, n_rows, n_chains, n_samples, probs, n_probs, *out, 0, g_create_error);
    if (cudaSetDevice(device) != cudaSuccess) { (void)cudaGetLastError(); g_create_error = "st_summarize_draws: cudaSetDevice failed"; return ST_ERR_CUDA; }
    const size_t per = (size_t)n_rows * n_samples, bytes = per * n_chains * sizeof(double);
    size_t fr = 0, tot = 0;
    if (cudaMemGetInfo(&fr, &tot) != cudaSuccess) { (void)cudaGetLastError(); g_create_error = "st_summarize_draws: cudaMemGetInfo failed"; return ST_ERR_CUDA; }
    // (the copy, plus the outputs' buffer and some headroom)
    const size_t need = bytes + (size_t)n_rows * (5 + n_probs) * sizeof(double) + (64u << 20);
    if (need > fr) {
      g_create_error = "st_summarize_draws: the draws need " + std::to_string(need) + " bytes of device memory and " + std::to_string(fr) +
                       " bytes are free";
      return ST_ERR_UNSUPPORTED;
    }
    double* d = nullptr;
    cudaError_t e = cudaMalloc((void**)&d, bytes);
    if (e != cudaSuccess) { (void)cudaGetLastError(); g_create_error = std::string("st_summarize_draws: ") + cudaGetErrorString(e); return ST_ERR_UNSUPPORTED; }
    e = cudaMemcpyAsync(d, draws, bytes, cudaMemcpyHostToDevice, 0);
    if (e == cudaSuccess) {
      std::vector<const double*> src(n_chains);
      for (int c = 0; c < n_chains; c++) src[c] = d + (size_t)c * per;
      rc = st::summarize_chains(src.data(), n_rows, n_chains, n_samples, probs, n_probs, *out, 0, g_create_error);
    } else {
      g_create_error = std::string("CUDA error in H2D draws: ") + cudaGetErrorString(e);
      rc = ST_ERR_CUDA;
    }
    cudaStreamSynchronize(0);
    cudaFree(d);
    return rc;
  } catch (const std::exception& ex) { g_create_error = ex.what(); } catch (...) { g_create_error = "unknown exception"; }
  return ST_ERR_INVALID;
}
// the checks st_fit_criteria and st_fit_criteria_integrated make of handle k (hk names it) against handle 0, whose store `which`
// holds S draws of n rows; *s: handle k's store
static int criteria_handle(const std::string& hk, st::Model& M0, const st_handle* hk_h, int which, int64_t n, int S,
                           const st::DrawStore::Store** s) {
  if (!hk_h) { M0.err = hk + " is NULL"; return ST_ERR_INVALID; }
  const st::Model& Mk = hk_h->model;
  if (Mk.device != M0.device) {
    M0.err = hk + " is on device " + std::to_string(Mk.device) + ", handle 0 on device " + std::to_string(M0.device);
    return ST_ERR_INVALID;
  }
  *s = Mk.store.find(which, hk + " has ", M0.err);
  if (!*s) return ST_ERR_INVALID;
  if ((*s)->n != n || (*s)->S != S) {
    M0.err = hk + " stores " + std::to_string((*s)->S) + " draws of " + std::to_string((*s)->n) + " rows, handle 0 " + std::to_string(S) +
             " draws of " + std::to_string(n) + " rows";
    return ST_ERR_INVALID;
  }
  if (Mk.p != M0.p || Mk.q != M0.q) {
    M0.err = hk + " has p = " + std::to_string(Mk.p) + ", q = " + std::to_string(Mk.q) + "; handle 0 p = " + std::to_string(M0.p) +
             ", q = " + std::to_string(M0.q);
    return ST_ERR_INVALID;
  }
  if (Mk.n_all != M0.n_all || std::memcmp(Mk.y.data(), M0.y.data(), M0.y.size() * sizeof(double)) ||
      std::memcmp(Mk.X.data(), M0.X.data(), M0.X.size() * sizeof(double)) ||
      std::memcmp(Mk.mv_id.data(), M0.mv_id.data(), M0.mv_id.size() * sizeof(int64_t))) {
    M0.err = hk + " has a different y, X or mv_id from handle 0 (the criteria compare fits of the same data)";
    return ST_ERR_INVALID;
  }
  return ST_OK;
}
// every store is complete before the kernel reads it on hs[0]'s stream
static int criteria_sync(const char* who, st_handle* const* hs, int32_t n_chains) {
  for (int k = 1; k < n_chains; k++)
    if (const cudaError_t e = cudaStreamSynchronize(hs[k]->model.stream)) {
      hs[0]->model.err = std::string(who) + ": CUDA error in sync of handle " + std::to_string(k) + ": " + cudaGetErrorString(e);
      return ST_ERR_CUDA;
    }
  return ST_OK;
}
int st_fit_criteria(st_handle* const* hs, int32_t n_chains, double r_eff, st_fit_criteria_out* out) {
  if (!hs || n_chains < 1 || !hs[0]) {  // (no handle to report to)
    g_create_error = n_chains < 1 ? "st_fit_criteria: n_chains must be at least 1" : "st_fit_criteria: hs or hs[0] is NULL";
    return ST_ERR_INVALID;
  }
  st_handle* h0 = hs[0];
  st::Model& M0 = h0->model;
  if (!out) { M0.err = "st_fit_criteria: out is NULL"; return ST_ERR_INVALID; }
  activate(h0);
  ST_GUARD_BEGIN
  const int64_t n = M0.store.get(0).n;
  const int S = M0.store.get(0).S, p = M0.p, q = M0.q;
  int rc = st::criteria_check("st_fit_criteria", n_chains, std::max(S, 1), r_eff, M0.err);
  if (rc) return rc;
  const size_t nb = (size_t)p * S * q, nt = (size_t)q * S, N = (size_t)n_chains * S;
  std::vector<const double*> src(n_chains);
  st::dvec beta(N * p * q), tausq(N * q);  // pooled draw g = k S + s: p x q, then q
  for (int k = 0; k < n_chains; k++) {
    const std::string hk = "st_fit_criteria: handle " + std::to_string(k);
    const st::DrawStore::Store* s = nullptr;
    rc = criteria_handle(hk, M0, hs[k], 0, n, S, &s);
    if (rc) return rc;
    const st::Model& Mk = hs[k]->model;
    const st::dvec& sm = Mk.store.samples;  // theta (npar x S) | beta (p x S x q) | tausq (q x S)
    if (sm.size() < nb + nt) { M0.err = hk + ": the stored run's beta / tausq samples are missing"; return ST_ERR_INVALID; }
    const double* be = sm.data() + (sm.size() - nb - nt);
    const double* ta = be + nb;
    for (int s2 = 0; s2 < S; s2++) {
      const size_t g = (size_t)k * S + s2;
      for (int j = 0; j < q; j++) {
        for (int a = 0; a < p; a++) beta[(g * q + j) * p + a] = be[a + (size_t)s2 * p + (size_t)j * p * S];
        tausq[g * q + j] = ta[j + (size_t)s2 * q];
      }
    }
    src[k] = s->d;
  }
  rc = criteria_sync("st_fit_criteria", hs, n_chains);
  if (rc) return rc;
  std::vector<char> obs(n);
  for (int64_t i = 0; i < n; i++) obs[i] = std::isfinite(M0.y[i]);
  const st::CritInputs in{M0.y.data(), M0.X.data(), M0.mv_id.data(), beta.data(), tausq.data(), p, q};
  return st::fit_criteria(src.data(), n, n_chains, S, r_eff, obs, &in, *out, M0.stream, M0.err);
  ST_GUARD_END(h0)
}
int st_fit_criteria_integrated(st_handle* const* hs, int32_t n_chains, double r_eff, st_fit_criteria_out* out) {
  if (!hs || n_chains < 1 || !hs[0]) {  // (no handle to report to)
    g_create_error = n_chains < 1 ? "st_fit_criteria_integrated: n_chains must be at least 1"
                                  : "st_fit_criteria_integrated: hs or hs[0] is NULL";
    return ST_ERR_INVALID;
  }
  st_handle* h0 = hs[0];
  st::Model& M0 = h0->model;
  if (!out) { M0.err = "st_fit_criteria_integrated: out is NULL"; return ST_ERR_INVALID; }
  activate(h0);
  ST_GUARD_BEGIN
  const int which = st::DrawStore::kLoglikInt;
  const int64_t n = M0.store.get(which).n;
  const int S = M0.store.get(which).S;
  int rc = st::criteria_check("st_fit_criteria_integrated", n_chains, std::max(S, 1), r_eff, M0.err);
  if (rc) return rc;
  std::vector<const double*> src(n_chains);
  for (int k = 0; k < n_chains; k++) {
    const st::DrawStore::Store* s = nullptr;
    rc = criteria_handle("st_fit_criteria_integrated: handle " + std::to_string(k), M0, hs[k], which, n, S, &s);
    if (rc) return rc;
    src[k] = s->d;
  }
  rc = criteria_sync("st_fit_criteria_integrated", hs, n_chains);
  if (rc) return rc;
  // the log-likelihood mode of fit_criteria_kernel: the stores hold ll itself, NaN at the rows whose y is missing
  std::vector<char> obs(n);
  for (int64_t i = 0; i < n; i++) obs[i] = std::isfinite(M0.y[i]);
  return st::fit_criteria(src.data(), n, n_chains, S, r_eff, obs, nullptr, *out, M0.stream, M0.err);
  ST_GUARD_END(h0)
}
int st_fit_criteria_loglik(int32_t device, const double* loglik, int64_t n_rows, int32_t n_chains, int32_t n_samples, double r_eff,
                           st_fit_criteria_out* out) {
  if (!out || n_rows < 0 || (n_rows > 0 && !loglik)) {
    g_create_error = "st_fit_criteria_loglik: out or loglik missing, or n_rows < 0";
    return ST_ERR_INVALID;
  }
  try {
    int rc = st::criteria_check("st_fit_criteria_loglik", n_chains, n_samples, r_eff, g_create_error);
    if (rc) return rc;
    // a row is unobserved when all its values are NaN; an observed row must be finite throughout
    const size_t per = (size_t)n_rows * n_samples, all = per * n_chains;
    std::vector<char> obs(n_rows);
    for (int64_t i = 0; i < n_rows; i++) obs[i] = !std::isnan(loglik[i]);
    for (size_t j = 0; j < all; j++) {
      const int64_t i = (int64_t)(j % n_rows);
      if (obs[i] ? !std::isfinite(loglik[j]) : !std::isnan(loglik[j])) {
        g_create_error = "st_fit_criteria_loglik: row " + std::to_string(i) + " is observed (not all NaN) but value " + std::to_string(j) +
                         " ([chain][sample][row] order) is not finite";
        return ST_ERR_INVALID;
      }
    }
    const bool any = out->lpd || out->elpd_loo || out->p_loo || out->pareto_k || out->elpd_waic || out->p_waic;
    if (!any || n_rows == 0) return st::fit_criteria(nullptr, n_rows, n_chains, n_samples, r_eff, obs, nullptr, *out, 0, g_create_error);
    if (cudaSetDevice(device) != cudaSuccess) { (void)cudaGetLastError(); g_create_error = "st_fit_criteria_loglik: cudaSetDevice failed"; return ST_ERR_CUDA; }
    const size_t bytes = all * sizeof(double);
    size_t fr = 0, tot = 0;
    if (cudaMemGetInfo(&fr, &tot) != cudaSuccess) { (void)cudaGetLastError(); g_create_error = "st_fit_criteria_loglik: cudaMemGetInfo failed"; return ST_ERR_CUDA; }
    // (the copy, plus the outputs' buffer and some headroom)
    const size_t need = bytes + (size_t)n_rows * 8 * sizeof(double) + (64u << 20);
    if (need > fr) {
      g_create_error = "st_fit_criteria_loglik: the log-likelihood needs " + std::to_string(need) + " bytes of device memory and " +
                       std::to_string(fr) + " bytes are free";
      return ST_ERR_UNSUPPORTED;
    }
    double* d = nullptr;
    cudaError_t e = cudaMalloc((void**)&d, bytes);
    if (e != cudaSuccess) { (void)cudaGetLastError(); g_create_error = std::string("st_fit_criteria_loglik: ") + cudaGetErrorString(e); return ST_ERR_UNSUPPORTED; }
    e = cudaMemcpyAsync(d, loglik, bytes, cudaMemcpyHostToDevice, 0);
    if (e == cudaSuccess) {
      std::vector<const double*> src(n_chains);
      for (int c = 0; c < n_chains; c++) src[c] = d + (size_t)c * per;
      rc = st::fit_criteria(src.data(), n_rows, n_chains, n_samples, r_eff, obs, nullptr, *out, 0, g_create_error);
    } else {
      g_create_error = std::string("CUDA error in H2D log-likelihood: ") + cudaGetErrorString(e);
      rc = ST_ERR_CUDA;
    }
    cudaStreamSynchronize(0);
    cudaFree(d);
    return rc;
  } catch (const std::exception& ex) { g_create_error = ex.what(); } catch (...) { g_create_error = "unknown exception"; }
  return ST_ERR_INVALID;
}
int st_bench_iteration(st_handle* h, const double* theta_prop, int do_swap, uint64_t seed, double* out3, float* ms_out) {
  if (!h || !theta_prop || !out3) return ST_ERR_INVALID;
  activate(h);
  ST_GUARD_BEGIN return h->model.bench_iteration(theta_prop, do_swap, seed, out3, ms_out);
  ST_GUARD_END(h)
}
int st_par_huvtransf_fwd(const double* par, int32_t npar, const double* bounds, double* out) {
  if (!par || !bounds || !out || npar < 0) return ST_ERR_INVALID;
  for (int j = 0; j < npar; j++) out[j] = st::mh_logit(par[j], bounds[j], bounds[j + npar]);
  return ST_OK;
}
int st_par_huvtransf_back(const double* par, int32_t npar, const double* bounds, double* out) {
  if (!par || !bounds || !out || npar < 0) return ST_ERR_INVALID;
  for (int j = 0; j < npar; j++) out[j] = st::mh_logistic(par[j], bounds[j], bounds[j + npar]);
  return ST_OK;
}
int st_mh_propose(int32_t npar, const double* param, const double* bounds, const double* paramsd, const double* U, double* out) {
  if (!param || !bounds || !paramsd || !U || !out || npar < 1 || npar > st::kMaxPar) return ST_ERR_INVALID;
  const bool oob = st::mh_propose(npar, param, bounds, paramsd, U, out);
  out[npar] = st::mh_jacobian(npar, out, param, bounds);
  out[npar + 1] = oob ? 1.0 : 0.0;
  return ST_OK;
}
int st_do_i_accept(double logaccept, double u) { return u < st::mh_accept_prob(logaccept) ? 1 : 0; }
int st_ram_adapt(int32_t npar, const double* metropolis_sd, int32_t steps, const double* U, const double* alpha, double* paramsd_out,
                 double* paramsd_trace) {
  if (!metropolis_sd || !paramsd_out || npar < 1 || npar > st::kMaxPar || steps < 0 || (steps > 0 && (!U || !alpha))) return ST_ERR_INVALID;
  try {
    const size_t pp = (size_t)npar * npar;
    std::vector<double> sd(pp), prod(pp), scratch(2 * pp);
    int started = 0;
    if (!st::ram_init(npar, metropolis_sd, sd.data(), prod.data())) return ST_ERR_INVALID;
    for (int m = 0; m < steps; m++) {
      st::ram_adapt(npar, sd.data(), prod.data(), &started, U + (size_t)m * npar, alpha[m], m, scratch.data());
      if (paramsd_trace) std::copy(sd.begin(), sd.end(), paramsd_trace + (size_t)m * pp);
    }
    std::copy(sd.begin(), sd.end(), paramsd_out);
    return ST_OK;
  } catch (...) {
    return ST_ERR_INVALID;
  }
}
int st_set_beta_index(st_handle* h, int faithful) {
  if (!h) return ST_ERR_INVALID;
  if (h->model.part && faithful) { h->model.err = "partitioned handles support only the corrected beta row index"; return ST_ERR_UNSUPPORTED; }
  activate(h);
  ST_GUARD_BEGIN return h->model.set_widx_mode(faithful != 0);
  ST_GUARD_END(h)
}
int st_nccl_unique_id(unsigned char* out128) {
  if (!out128) return ST_ERR_INVALID;
  std::string e;
  const int rc = st::Model::nccl_unique_id(out128, e);
  if (rc) g_create_error = e;
  return rc;
}
int st_attach_nccl(st_handle* h, const unsigned char* id128) {
  if (!h || !id128) return ST_ERR_INVALID;
  activate(h);
  return h->model.attach_nccl(id128);
}
int st_get_counters(st_handle* h, double* out8) {
  if (!h || !out8) return ST_ERR_INVALID;
  out8[0] = h->model.n_launches; out8[1] = h->model.f_alg; out8[2] = h->model.f_exec; out8[3] = h->model.n_cov;
  out8[4] = h->model.f_alg_build; out8[5] = h->model.f_exec_build; out8[6] = h->model.b_alg_build; out8[7] = (double)sizeof(st::ChainDev);
  return ST_OK;
}
int st_sync(st_handle* h) {
  if (!h) return ST_ERR_INVALID;
  activate(h);
  return h->model.sync();
}

// ---- DAG construction
int st_kthresholds(const double* x, int64_t n, int32_t k, double* res) {
  if (!x || n <= 0 || k < 1 || (k > 1 && !res)) return ST_ERR_INVALID;
  try { st::kthresholds(x, n, k, res); } catch (...) { return ST_ERR_INVALID; }
  return ST_OK;
}
int st_part_axis_parallel_lmt(const double* coords, int64_t n, int32_t d, const double* thr, const int64_t* thr_ptr, double* out) {
  if (!coords || !thr_ptr || !out) return ST_ERR_INVALID;
  try { st::part_axis_parallel_lmt(coords, n, d, thr, thr_ptr, out); } catch (...) { return ST_ERR_INVALID; }
  return ST_OK;
}
int st_number_revalue(const int64_t* orig, int64_t nr, int32_t nc, const int64_t* from_val, const int64_t* to_val, int64_t nfrom, int64_t* out) {
  if (!orig || !out) return ST_ERR_INVALID;
  try { st::number_revalue(orig, nr, nc, from_val, to_val, nfrom, out); } catch (...) { return ST_ERR_INVALID; }
  return ST_OK;
}
int st_make_edges(const double* parchimat, int64_t nr, int32_t L, const int64_t* non_empty_blocks, int64_t n_ne,
                  const int64_t* res_is_ref, int32_t limited, int64_t* par_ptr, int64_t* par_idx, int64_t* chi_ptr,
                  int64_t* chi_idx, int64_t* counts) {
  if (!parchimat || !res_is_ref || !counts || L < 1) return ST_ERR_INVALID;
  try {
    st::CSR par, chi;
    int64_t nb = 0;
    st::make_edges(parchimat, nr, L, non_empty_blocks, n_ne, res_is_ref, limited != 0, par, chi, nb);
    counts[0] = nb; counts[1] = (int64_t)par.idx.size(); counts[2] = (int64_t)chi.idx.size();
    if (par_idx) {
      std::copy(par.ptr.begin(), par.ptr.end(), par_ptr);
      std::copy(par.idx.begin(), par.idx.end(), par_idx);
      std::copy(chi.ptr.begin(), chi.ptr.end(), chi_ptr);
      std::copy(chi.idx.begin(), chi.idx.end(), chi_idx);
    }
  } catch (...) { return ST_ERR_INVALID; }
  return ST_OK;
}

int st_make_tree(const st_tree_opts* o, st_tree** out) {
  if (!o || !out || !o->coords || !o->y || !o->mv_id || o->n_all <= 0) return ST_ERR_INVALID;
  *out = nullptr;
  try {
    st_tree* t = new st_tree();
    std::string e;
    if (!st::make_tree(o->coords, o->y, o->mv_id, o->n_all, o->cell_size, o->K[0], o->K[1], o->start_level, o->tree_depth,
                       o->last_not_reference != 0, o->cherrypick_same_margin != 0, o->cherrypick_group_locations != 0,
                       o->seed, t->t, e)) {
      g_create_error = e;
      delete t;
      return ST_ERR_INVALID;
    }
    *out = t;
  } catch (const std::exception& ex) { g_create_error = ex.what(); return ST_ERR_INVALID; } catch (...) { return ST_ERR_INVALID; }
  return ST_OK;
}
void st_tree_destroy(st_tree* t) { delete t; }
int st_tree_attach(const st_tree* t, int64_t n_new, const double* coords_new, const int64_t* mv_new, int32_t limited,
                   int64_t* group, int64_t* par_ptr, int64_t* par_idx, int64_t* counts) {
  if (!t || !counts || n_new < 0 || (n_new > 0 && (!coords_new || !mv_new))) return ST_ERR_INVALID;
  try {
    st::ivec g;
    st::CSR par;
    std::string e;
    if (!st::tree_attach(t->t, coords_new, mv_new, n_new, limited != 0, g, par, e)) { g_create_error = e; return ST_ERR_INVALID; }
    counts[0] = (int64_t)par.ptr.size() - 1; counts[1] = (int64_t)par.idx.size();
    if (par_idx) {
      if (!group || !par_ptr) return ST_ERR_INVALID;
      std::copy(g.begin(), g.end(), group);
      std::copy(par.ptr.begin(), par.ptr.end(), par_ptr);
      std::copy(par.idx.begin(), par.idx.end(), par_idx);
    }
  } catch (const std::exception& ex) { g_create_error = ex.what(); return ST_ERR_INVALID; } catch (...) { return ST_ERR_INVALID; }
  return ST_OK;
}
int st_tree_sizes(const st_tree* t, int64_t* o) {
  if (!t || !o) return ST_ERR_INVALID;
  o[0] = t->t.n_blocks; o[1] = (int64_t)t->t.res_is_ref.size(); o[2] = t->t.parchi_rows; o[3] = t->t.parchi_cols;
  o[4] = (int64_t)t->t.parents.idx.size(); o[5] = (int64_t)t->t.children.idx.size();
  return ST_OK;
}
int st_tree_get(const st_tree* t, int64_t* blocking, int64_t* res, int64_t* res_is_ref, double* parchimat,
                int64_t* indexing_ptr, int64_t* indexing_idx, int64_t* parents_ptr, int64_t* parents_idx,
                int64_t* children_ptr, int64_t* children_idx, double* block_names, double* block_groups) {
  if (!t) return ST_ERR_INVALID;
  const st::TreeResult& T = t->t;
  auto cp = [](const auto& v, auto* dst) { if (dst) std::copy(v.begin(), v.end(), dst); };
  cp(T.blocking, blocking); cp(T.res, res); cp(T.res_is_ref, res_is_ref); cp(T.parchimat, parchimat);
  cp(T.indexing.ptr, indexing_ptr); cp(T.indexing.idx, indexing_idx);
  cp(T.parents.ptr, parents_ptr); cp(T.parents.idx, parents_idx);
  cp(T.children.ptr, children_ptr); cp(T.children.idx, children_idx);
  cp(T.block_names, block_names); cp(T.block_groups, block_groups);
  return ST_OK;
}

int st_cross_covariance_ag10(const double* coords1, const int64_t* mv1, int64_t n1, const double* coords2, const int64_t* mv2,
                             int64_t n2, const double* ai1, const double* ai2, const double* phi_i, const double* thetamv,
                             int32_t n_thetamv, const double* Dmat, int32_t q, int32_t device, double* out) {
  if (!coords1 || !coords2 || !mv1 || !mv2 || !out || q < 2 || q > st::kMaxQ) {
    g_create_error = "Invalid Dmat for multivariate data";  // covariance_functions.cpp:317-319
    return ST_ERR_INVALID;
  }
  try {
    // pack (ai1, ai2, phi_i, thetamv, lower triangle of Dmat) in the theta layout and reuse make_covtab
    const int n_cbase = q > 2 ? 3 : 1;
    if (n_thetamv < n_cbase) return ST_ERR_INVALID;
    st::dvec th;
    th.insert(th.end(), ai1, ai1 + q); th.insert(th.end(), ai2, ai2 + q); th.insert(th.end(), phi_i, phi_i + q);
    th.insert(th.end(), thetamv, thetamv + n_cbase);
    for (int j = 0; j < q; j++)
      for (int i = j + 1; i < q; i++) th.push_back(Dmat[i + (size_t)j * q]);
    st::CovTab tab;
    std::string e;
    if (!st::make_covtab(th.data(), (int)th.size(), q, tab, e)) { g_create_error = e; return ST_ERR_INVALID; }
    if (cudaSetDevice(device) != cudaSuccess) { g_create_error = "cudaSetDevice failed"; return ST_ERR_CUDA; }
    std::vector<int> q1(n1), q2(n2);
    for (int64_t i = 0; i < n1; i++) q1[i] = (int)mv1[i] - 1;
    for (int64_t i = 0; i < n2; i++) q2[i] = (int)mv2[i] - 1;
    for (int v : q1) if (v < 0 || v >= q) { g_create_error = "mv_id outside 1..q"; return ST_ERR_INVALID; }
    for (int v : q2) if (v < 0 || v >= q) { g_create_error = "mv_id outside 1..q"; return ST_ERR_INVALID; }
    double *dx1 = nullptr, *dx2 = nullptr, *dout = nullptr;
    int *dq1 = nullptr, *dq2 = nullptr;
    cudaError_t ce = cudaSuccess;
    auto chk = [&](cudaError_t c) { if (ce == cudaSuccess) ce = c; };
    chk(cudaMalloc((void**)&dx1, 2 * n1 * sizeof(double)));
    chk(cudaMalloc((void**)&dx2, 2 * n2 * sizeof(double)));
    chk(cudaMalloc((void**)&dq1, n1 * sizeof(int)));
    chk(cudaMalloc((void**)&dq2, n2 * sizeof(int)));
    chk(cudaMalloc((void**)&dout, (size_t)n1 * n2 * sizeof(double)));
    if (ce == cudaSuccess) {
      chk(cudaMemcpy(dx1, coords1, 2 * n1 * sizeof(double), cudaMemcpyHostToDevice));
      chk(cudaMemcpy(dx2, coords2, 2 * n2 * sizeof(double), cudaMemcpyHostToDevice));
      chk(cudaMemcpy(dq1, q1.data(), n1 * sizeof(int), cudaMemcpyHostToDevice));
      chk(cudaMemcpy(dq2, q2.data(), n2 * sizeof(int), cudaMemcpyHostToDevice));
      chk(st::launch_crosscov(dx1, dx1 + n1, dq1, n1, dx2, dx2 + n2, dq2, n2, tab, dout, 0));
      chk(cudaMemcpy(out, dout, (size_t)n1 * n2 * sizeof(double), cudaMemcpyDeviceToHost));
    }
    cudaFree(dx1); cudaFree(dx2); cudaFree(dq1); cudaFree(dq2); cudaFree(dout);
    if (ce != cudaSuccess) { g_create_error = std::string("CUDA error: ") + cudaGetErrorString(ce); return ST_ERR_CUDA; }
  } catch (...) { return ST_ERR_INVALID; }
  return ST_OK;
}

}  // extern "C"
