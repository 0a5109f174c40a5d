// st_mcmc.cpp — the MCMC driver: same control flow as spamtree_mv_mcmc (spamtree_fit.cpp:5-430), calling the model
// layer through the reference-named operations.  Printing and R's interrupt polling have no counterpart here.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>

#include "../../include/spamtree_b200.h"
#include "st_mh.hpp"
#include "st_model.hpp"

namespace st {

// Robust adaptive Metropolis (Vihola 2012) as the reference runs it, mh_adapt.h:40-135: state of st_mh.hpp's functions
struct RAMAdapt {
  int p = 0, started = 0;
  dvec paramsd, prodparam, scratch;
  bool init(int npars, const double* metropolis_sd) {
    p = npars;
    paramsd.assign((size_t)p * p, 0.0); prodparam.assign((size_t)p * p, 0.0); scratch.assign(2 * (size_t)p * p, 0.0);
    return ram_init(p, metropolis_sd, paramsd.data(), prodparam.data());
  }
  bool adapt(const dvec& U, double alpha, int mc) { return ram_adapt(p, paramsd.data(), prodparam.data(), &started, U.data(), alpha, mc, scratch.data()); }
};

int mcmc_run(Model& M, const st_mcmc_opts& o, st_mcmc_out& out) {
  // rng_mode 1: the device-resident chain — proposal, accept decision, RAM adaptation, tausq / beta draws and yhat on the
  // device, no host round trip per iteration (st_model.cu: Model::chain_run)
  if (o.rng_mode == 1) return M.chain_run(o, out);
  if (M.keep_mask) {
    M.err = "st_mcmc_run: the device sample store (st_keep_samples_on_device) needs the device-resident chain (rng_mode = 1)";
    return ST_ERR_UNSUPPORTED;
  }
  // rng_mode 0: every draw from one host stream, in the reference's order (lock-step with the oracle and with the
  // reference's own driver); a partitioned run draws for every row of the whole problem on every rank and keeps its own
  if (M.part && M.global_rows.empty()) {
    M.err = "partitioned handle without global_rows: the host random stream (rng_mode 0) would differ between the ranks";
    return ST_ERR_INVALID;
  }
  M.rng.seed(o.seed);
  double o3[3];
  int rc = M.get_loglik_comps_w(0, o3);  // spamtree_fit.cpp:110-111
  if (rc) return rc;
  rc = M.get_loglik_comps_w(1, o3);
  if (rc) return rc;
  const int npar = (int)M.theta[M.cur].size();
  dvec param = M.theta[M.cur], predict_param = param;
  double current_loglik = M.loglik_w[M.cur];
  const int mcmc = o.thin * o.keep + o.burn;
  if (npar > kMaxPar) { M.err = "more than 64 covariance parameters"; return ST_ERR_UNSUPPORTED; }
  RAMAdapt ad;
  if (!ad.init(npar, o.mcmcsd)) {  // arma::chol(S, "lower") throws in the reference (mh_adapt.h:86)
    M.err = "mcmcsd is not positive definite";
    return ST_ERR_INVALID;
  }
  int msaved = 0;
  out.n_accepted = out.n_chol_fail = 0;
  dvec zbuf, wbuf, xbbuf, zglob;
  zbuf.resize(M.n_all);
  const bool pglob = M.part && !M.global_rows.empty();  // partitioned: draw for every row of the problem, keep ours
  if (pglob) zglob.resize(M.n_global_rows);
  // w of a saved iteration goes to the caller's buffer asynchronously (overlapping the next iteration) unless yhat, which
  // is formed on the host from w, is requested too
  const bool async_save = out.w_mcmc && !out.yhat_mcmc;
  CopyOut co(M.stream, M.copy_stream, M.err);
  if (async_save) { rc = co.open({out.w_mcmc}, (size_t)o.keep * M.n_all * sizeof(double), 1, M.n_all); if (rc) return rc; }
  // ST_PROFILE_MCMC=1: host wall-clock per phase of the loop, printed by every rank at the end (development aid)
  static const bool prof = getenv("ST_PROFILE_MCMC") != nullptr;
  double tph[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  auto tick = [&]() { return std::chrono::steady_clock::now(); };
  auto lap = [&](int i, std::chrono::steady_clock::time_point& t) {
    if (!prof) return;
    const auto n = tick();
    tph[i] += std::chrono::duration<double>(n - t).count();
    t = n;
  };
  const auto t0 = std::chrono::steady_clock::now();
  for (int m = 0; m < mcmc; m++) {
    auto tl = tick();
    bool predicting = false;
    const int mx = m - o.burn;
    if (mx >= 0 && mx % o.thin == 0) predicting = true;
    if (o.sample_w) {  // :183-187
      if (pglob) {
        for (int64_t i = 0; i < M.n_global_rows; i++) zglob[i] = M.rng.norm();
        for (int64_t i = 0; i < M.n_all; i++) zbuf[i] = zglob[M.global_rows[i]];
      } else {
        for (int64_t i = 0; i < M.n_all; i++) zbuf[i] = M.rng.norm();  // bigrnorm (:1018)
      }
      rc = M.deal_with_w(zbuf.data(), 0);
      if (rc) return rc;
      lap(0, tl);
      double o2[2];
      rc = M.get_loglik_w(0, o2);
      if (rc) return rc;
      current_loglik = M.loglik_w[M.cur];
      lap(1, tl);
    }
    if (o.sample_theta) {  // :203-289
      dvec U(npar), new_param(npar);
      for (int j = 0; j < npar; j++) U[j] = M.rng.norm();
      mh_propose(npar, param.data(), o.set_unif_bounds, ad.paramsd.data(), U.data(), new_param.data());  // :211-215
      M.theta_update(1, new_param.data());
      rc = M.get_loglik_comps_w(1, o3);
      if (rc) return rc;
      lap(2, tl);
      const bool acceptable = o3[2] != 0.0;
      const double new_loglik = M.loglik_w[1 - M.cur];
      current_loglik = M.loglik_w[M.cur];
      if (std::isnan(current_loglik)) { M.err = "At nan loglik: error."; return ST_ERR_NAN; }
      const double jac = mh_jacobian(npar, new_param.data(), param.data(), o.set_unif_bounds);  // mh_adapt.h:230-239
      const double logaccept = new_loglik - current_loglik + jac;
      const double acceptj = mh_accept_prob(logaccept);  // do_I_accept, mh_adapt.h:20-36
      const double u = M.rng.unif();
      const bool accepted = (u < acceptj) && acceptable;
      if (!acceptable) out.n_chol_fail++;
      if (accepted) {
        out.n_accepted++;
        current_loglik = new_loglik;
        M.accept_make_change();
        param = new_param;
      }
      // (a failed chol(S) keeps the previous factor; the reference's arma::chol would throw and end the run, mh_adapt.h:133)
      if (o.adapting) ad.adapt(U, (acceptable ? 1.0 : 0.0) * std::exp(logaccept), m);  // :285
      lap(3, tl);
    }
    bool need_update = false;  // :300
    for (int j = 0; j < npar; j++)
      if (std::fabs(param[j] - predict_param[j]) > 1e-05) need_update = true;
    if (predicting && o.sample_predicts && o.sample_w) {
      rc = M.predict(need_update);
      if (rc) return rc;
      predict_param = param;
    }
    lap(4, tl);
    if (o.sample_tausq) { rc = M.gibbs_sample_tausq(nullptr); if (rc) return rc; }
    if (o.sample_beta) { rc = M.gibbs_sample_beta(nullptr, o.faithful_beta_index != 0); if (rc) return rc; }
    lap(5, tl);
    if (mx >= 0 && mx % o.thin == 0) {  // save, :376-389
      if (out.tausq_mcmc)
        for (int j = 0; j < M.q; j++) out.tausq_mcmc[j + (size_t)msaved * M.q] = 1.0 / M.tausq_inv[j];
      if (out.beta_mcmc)
        for (int j = 0; j < M.q; j++)
          for (int a = 0; a < M.p; a++)
            out.beta_mcmc[a + (size_t)msaved * M.p + (size_t)j * M.p * o.keep] = M.Bcoeff[a + (size_t)j * M.p];
      if (out.theta_mcmc)
        for (int j = 0; j < npar; j++) out.theta_mcmc[j + (size_t)msaved * npar] = M.theta[M.cur][j];
      const bool want_rows = (out.w_mcmc || out.yhat_mcmc) && !async_save;
      if (async_save) { rc = M.save_rows(co, 0, nullptr, out.w_mcmc + (size_t)msaved * M.n_all); if (rc) return rc; }
      if (want_rows) {
        wbuf.resize(M.n_all);
        rc = M.get_w(wbuf.data());
        if (rc) return rc;
        if (out.w_mcmc) std::copy(wbuf.begin(), wbuf.end(), out.w_mcmc + (size_t)msaved * M.n_all);
      }
      if (out.yhat_mcmc) {
        xbbuf.resize(M.n_all);
        rc = M.get_xb(xbbuf.data());
        if (rc) return rc;
      }
      // arma::randn(n) of :384 — drawn whether or not yhat is kept, and for every row of the whole problem on every rank of
      // a partition, so that the one host stream stays in step everywhere
      if (pglob)
        for (int64_t i = 0; i < M.n_global_rows; i++) zglob[i] = M.rng.norm();
      for (int64_t i = 0; i < M.n_all; i++) {
        const double e = pglob ? zglob[M.global_rows[i]] : M.rng.norm();
        if (out.yhat_mcmc)
          out.yhat_mcmc[i + (size_t)msaved * M.n_all] = xbbuf[i] + wbuf[i] + std::pow(M.tausq_inv[M.mv_id[i] - 1], -.5) * e;
      }
      msaved++;
    }
    lap(6, tl);
  }
  rc = co.finish();  // the timed region ends when every saved w is on the host
  if (rc) return rc;
  out.mcmc_time = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  if (prof)
    fprintf(stderr, "[mcmc profile] rank %d: %d iterations, %lld accepted; ms/iteration: gibbs %.3f llw %.3f build %.3f accept+adapt %.3f predict %.3f tausq+beta %.3f save %.3f | total %.3f\n",
            M.rank, mcmc, (long long)out.n_accepted, 1e3 * tph[0] / mcmc, 1e3 * tph[1] / mcmc, 1e3 * tph[2] / mcmc, 1e3 * tph[3] / mcmc,
            1e3 * tph[4] / mcmc, 1e3 * tph[5] / mcmc, 1e3 * tph[6] / mcmc, 1e3 * out.mcmc_time / mcmc);
  if (out.paramsd) std::copy(ad.paramsd.begin(), ad.paramsd.end(), out.paramsd);
  return 0;
}

}  // namespace st
