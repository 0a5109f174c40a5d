// st_kernels.cuh — launch wrappers of the sm_100a kernels in st_kernels.cu (host-callable; no kernel types leak out)
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

#include "st_build_plan.cuh"
#include "st_model.hpp"

namespace st {

constexpr int kGibbsThreads = 64;   // two warps per block (measured on C4: 128 -> 1.46 ms, 64 -> 1.14 ms, 32 -> 1.21 ms per sweep)
constexpr int kGramThreads = 256;
constexpr int kGramMaxRows = 256;   // rows gram_level_kernel stages per chunk
constexpr int kGramChildTab = 256;  // (child, tile) offsets it tabulates
constexpr int kGramFusedTab = 64;   // children whose row blocks it tabulates
constexpr int kLlwThreads = 128;
constexpr int kLlwMaxP = 1024;  // parent-set rows the LLW kernel stages per warp (checked at st_create)
constexpr double kHl2pi = -0.91893853320467274178;  // -0.5 * log(2 pi)  (spamtree_model.h:20)

inline size_t gibbs_smem_bytes(int is_ref, int m, int P, int k) {
  const size_t msq = is_ref ? (size_t)m * tile_rs(m) + (size_t)m * m : 2 * (size_t)m;
  return 8 * (msq + (size_t)P + (size_t)(k + 1) * m + 3 * (size_t)m) + 16;
}

// Opts a kernel in to `smem` bytes of dynamic shared memory on the CURRENT device if it has not been opted in to at
// least that much there yet (the attribute is per device; static + dynamic together exceed the default 48 KB long before
// the dynamic part alone does, so the opt-in is unconditional).  `table` is the caller's per-kernel cache.
struct SmemOptIn { size_t configured[64] = {}; };
template <class K>
inline cudaError_t ensure_dynamic_smem(K kern, size_t smem, SmemOptIn& table) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= 64) return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (smem <= table.configured[dev]) return cudaSuccess;
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess) table.configured[dev] = smem;
  return e;
}

// Slot arguments: `D` holds both theta-slots and the device chain state; `rel` = 0 selects param_data, 1 alter_data
// (the kernel reads chain->cur).  `run_flag` (or NULL): device int, the launch is a no-op when it is 0.
// mode 0 / 1: reference / non-reference level of the slot; mode 2: prediction blocks (predG = Hpred receives H, predRi = sd);
// mode 3: forward-only prediction of new rows (predG receives mean = K_{u,pa} K_pa^-1 w_pa, predRi sd, both at rioff).
cudaError_t launch_build(int mode, const DevTree& T, const DevSlots& D, int rel, double* predG, double* predRi, int want_H,
                         const int* grp_slot0, const int* grp_nn, int ngrp, const double* w, int* fail, int ns, int phase, size_t smem,
                         cudaStream_t st, int nthreads, unsigned long long* prof = nullptr, bool pdl = false,
                         const int* run_flag = nullptr);  // pdl: programmatic dependent launch on the previous kernel of the stream
cudaError_t launch_gibbs(int is_ref, const DevTree& T, const DevSlots& D, int slot0, int nslots, double* w,
                         const double* xb, const double* z, const double* tausq_inv, const double* SigS, double* V,
                         double* probe_sig, double* probe_smu, int* fail, size_t smem, cudaStream_t st, bool pdl = false,
                         double* ll = nullptr,   // ll != NULL: the ILOO variant, integrated log-likelihood into ll (node-major) at
                         const double* yobs = nullptr);  // the rows where yobs (y node-major, NaN: not observed) is not NaN
cudaError_t launch_gram(const DevTree& T, const DevSlots& D, int slot0, int nslots, double* U, double* SigS, int rch,
                        int ldx, int tile_doubles, int stage_off, int threads, cudaStream_t st, const int* run_flag = nullptr,
                        bool pdl = false);  // pdl: only after another gram launch (the kernel waits before it reads the children's tiles only)
// blocks [slot0, slot0 + nslots) of the slot.  vrow (or NULL): per row of a reference block, s_r = ([G | -Ri] [w_pa ; w_u])_r =
// -(L^-1 w)_r is stored as well; parked = 1: the blocks are childless non-reference blocks whose storage still holds the
// unscaled Z of the forward half of BUILD (st_build.cu) — their log-density pieces are formed from Z and the v = L^-1 w_pa read
// off vrow (the ancestors must have been through a vrow pass)
cudaError_t launch_llw(const DevTree& T, const DevSlots& D, int rel, int slot0, int nslots, const double* w, int maxlen, cudaStream_t st,
                       double* vrow = nullptr, int parked = 0);
// out8[0..2] = {sum logdet + sum llcomp, sum logdet, 0} over blocks [0, n_top) and out8[4..6] = the same over [n_top, n) with
// out8[6] = *fail (or 0): the two parts a partitioned run needs (replicated blocks once, the rank's own all-reduced)
// scratch: kReduceScratch doubles (partial sums + two counters that must start at zero), private to the stream
constexpr int kReduceScratch = 4 * 32 + 2;
cudaError_t launch_loglik_reduce(const DevSlots& D, int rel, int n_top, int n, int* fail, double* out8, double* scratch,
                                 cudaStream_t st);
cudaError_t launch_frontier_sum(const DevTree& T, int n, const int* pseudo, const int* c0, const int* c1, const int* vlen,
                                const int* ulen, double* V, double* U, int do_v, int do_u, cudaStream_t st);
cudaError_t launch_predict_sample(const DevTree& T, int slot0, int nslots, const double* Hpred, const double* sdpred,
                                  double* w, const double* z, cudaStream_t st);
// z[i] = N(0,1) from Philox keyed by (seed, rowkey[i], counter + *iter_ptr): rowkey = the row's id in the whole problem, so
// that a partitioned run draws the same number for the same row whatever the number of ranks
cudaError_t launch_normals(double* z, long long n, uint64_t seed, uint64_t counter, const long long* rowkey, const int* iter_ptr,
                           cudaStream_t st);
cudaError_t launch_rowstats(const DevTree& T, const int* widx, long long n_all, int p, int q, const double* w,
                            const double* xb, double* partial, int nblocks, double* out, cudaStream_t st);
cudaError_t launch_xb(const DevTree& T, long long n_all, int p, const double* bcoeff, double* xb, cudaStream_t st);
cudaError_t launch_permute(const double* src, double* dst, const long long* map, long long n, cudaStream_t st);
cudaError_t launch_crosscov(const double* x1, const double* y1, const int* q1, long long n1, const double* x2,
                            const double* y2, const int* q2, long long n2, const CovTab& tab, double* out,
                            cudaStream_t st);
// ---- the device-resident chain (st_chain.hpp): one tiny kernel per step of spamtree_fit.cpp:203-289 / :376-389
// proposal: U ~ N(0, I) (Philox), theta' = back(fwd(theta) + paramsd U) into the alter slot's theta, its covariance table
cudaError_t launch_mh_propose(ChainDev* C, cudaStream_t st, int iter_offset = 0);  // 1: the next iteration's proposal (after accept, before the tick)
// accept step.  mode 0: Metropolis rule (Jacobian, uniform draw, RAM adaptation); 1: take the proposal if BUILD succeeded;
// 2: reject (1 / 2: bench hooks).  have_llw: red_llw holds the log-density of the current slot at the new w.
cudaError_t launch_mh_accept(ChainDev* C, int mode, int have_llw, cudaStream_t st, int npar = 0);  // npar: stages the adaptation in shared memory
// need_update of spamtree_fit.cpp:300 -> C->predict_build; predict_param <- theta
cudaError_t launch_predict_gate(ChainDev* C, cudaStream_t st);
// gibbs_sample_tausq (:1393-1417) then gibbs_sample_beta (:1364-1391) from the statistics of rowstats_kernel, random
// numbers from Philox; scratch: q * 3 * p * p doubles
cudaError_t launch_tausq_beta(ChainDev* C, const double* stats, const double* xtx, double* tausq_inv, double* bcoeff,
                              double* scratch, int sample_tausq, int sample_beta, cudaStream_t st, int p = 0, int q = 0);
// the saved iteration's theta / beta / tausq into the device sample arrays (layouts of st_mcmc_out), then C->msaved++
cudaError_t launch_record(ChainDev* C, const double* tausq_inv, const double* bcoeff, double* theta_mcmc, double* beta_mcmc,
                          double* tausq_mcmc, int keep, cudaStream_t st, int tick = 0);  // tick: also advances the iteration counter
// yhat = XB + w + tausq^(1/2) N(0,1) in boundary order (spamtree_fit.cpp:384)
cudaError_t launch_yhat(const DevTree& T, const double* w, const double* xb, const double* tausq_inv, const long long* iperm,
                        const long long* rowkey, long long n, const ChainDev* C, double* out, cudaStream_t st);
cudaError_t launch_chain_tick(ChainDev* C, cudaStream_t st);  // iter++
// host-driven path: theta and its covariance table into the slot `rel` (0 param_data, 1 alter_data) — passed by value as
// kernel parameters, so no host buffer has to outlive the call and nothing synchronises; flip: accept_make_change
struct ThetaPack {
  int n;
  double theta[kMaxPar];
  CovTab tab;
};
cudaError_t launch_chain_set_theta(ChainDev* C, int rel, const ThetaPack& pack, cudaStream_t st);
cudaError_t launch_chain_flip(ChainDev* C, cudaStream_t st);
// ---- predict_new (Model::predict_new)
// dst[i] = src[perm[i] * si + b * sb]: sample b of a staged block of samples, boundary order -> node-major order
cudaError_t launch_gather_sample(const double* src, long long si, long long sb, int b, const long long* perm, double* dst, long long n,
                                 cudaStream_t st);
struct PredDrawPack {
  double beta[kMaxStats];  // p x q of the sample
  double sdtau[kMaxQ];     // sqrt(tausq) per outcome
};
// draws of sample j (position in the call) at n new rows: layout position k (mean / sd) -> caller row lay2row[k] (mvq, X
// (n x p, column-major, or NULL), z / eps (or NULL: Philox keyed by (seed, row, j)), outputs, acc: 4 doubles per row)
cudaError_t launch_predict_draw(long long n, const long long* lay2row, const int* mvq, const double* X, int p, const double* mean,
                                const double* sd, const PredDrawPack& pk, uint64_t seed, int j, const double* z, const double* eps,
                                double* wout, double* yout, double* mout, double* sdout, double* acc, cudaStream_t st);
// out4 = {mean w, sd w, mean y, sd y} (n each) from acc after S samples
cudaError_t launch_predict_moments(long long n, int S, const double* acc, double* out4, cudaStream_t st);
// ---- per-row summaries of a [sample][row] store of S draws of n rows (st_summarize; DESIGN.md §5c)
constexpr int kSummaryThreads = 512;
constexpr int kSummaryMaxRows = 32;   // rows one CTA stages at most (the tile shape at small S)
// rows per CTA for S draws in smem_cap bytes of shared memory: the largest power of two <= kSummaryMaxRows whose keys fit;
// 0 when not even one row fits
int summary_rows_per_cta(int S, size_t smem_cap);
size_t summary_smem_bytes(int S, int R);
// mean, sd (ddof 1), quant (n x np, column-major; numpy's "linear" quantiles of probs[np], a device array), mcse and ess
// (batch means); every output a device array of n (quant: n np)
cudaError_t launch_summary(const double* src, long long n, int S, int R, const double* probs, int np, double* mean, double* sd, double* quant,
                           double* mcse, double* ess, cudaStream_t st);
// ---- K chains of S draws of n rows, chain c's draw (s, i) at src[c][s * n + i] (src: a device array of K device pointers):
// pooled mean, sd (ddof 1), quantiles, and rank-normalised split-R-hat, bulk-ESS and tail-ESS (st_summarize_chains; §5d).
// Shared memory per row: 2 K S keys and 2 K doubles, so one row fits while K (S + 1) <= (smem_cap - 8 kSummaryThreads) / 16
size_t chains_smem_bytes(int K, int S, int R);
int chains_rows_per_cta(int K, int S, size_t smem_cap);  // as summary_rows_per_cta; 0 when not even one row fits
cudaError_t launch_chains_summary(const double* const* src, long long n, int K, int S, int R, const double* probs, int np, double* mean,
                                  double* sd, double* quant, double* rhat, double* ess_bulk, double* ess_tail, cudaStream_t st);
// ---- model criteria over K chains of S draws of n rows (st_fit_criteria, st_fit_criteria_loglik; DESIGN.md §5e).  Shared
// memory as summary_kernel's with N = K S draws per row: R = summary_rows_per_cta(K S, cap) rows per CTA.
struct CritParams {
  const double* y;      // n, NaN: unobserved row.  NULL: the draws are the log-likelihood itself (NaN in draw 0: unobserved)
  const double* X;      // n x p, column-major
  const int* mvq;       // n, 0-based outcome
  const double* beta;   // draw g's p x q coefficients at beta[g p q ..), column-major
  const double* tausq;  // draw g's q variances at tausq[g q ..)
  const double* bbar;   // p x q pooled posterior means
  const double* tbar;   // q
  int p, q;
};
int criteria_tail_len(int N, double r_eff);  // min(ceil(0.2 N), ceil(3 sqrt(N / r_eff))), as R loo's n_pareto_draws
// out: 8 n doubles, [lpd | elpd_loo | p_loo | pareto_k | elpd_waic | p_waic | -2 mean ll | -2 log N(y; plug-in means)]
cudaError_t launch_fit_criteria(const double* const* src, long long n, int K, int S, int R, double r_eff, const CritParams& P, double* out,
                                cudaStream_t st);

}  // namespace st
