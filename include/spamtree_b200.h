/* spamtree_b200.h — C ABI of libspamtree_b200.so
 *
 * Drop-in boundary for the per-iteration MCMC hot path of SpamTrees (reference:
 * mkln/spamtree v0.2.1).  Every entry point below replaces one piece of the
 * reference's Rcpp/C++ model layer; the reference interface it stands in for is
 * cited as file:line (paths relative to the reference tree).  Plain pointers and
 * sizes only; no C++ exceptions cross this boundary; every function returns an
 * st_status (0 = ok) unless stated otherwise.  All matrices are FP64 COLUMN-MAJOR
 * (as arma::mat), all row ids / block ids 0-based unless stated otherwise, rows in
 * the caller's ("boundary") order — the order spamtree() passes to
 * spamtree_mv_mcmc (R/spamtree_fit.R:267-269, :327-362).
 *
 * Not re-entrant per handle.  One host thread drives one GPU per handle.
 */
#ifndef SPAMTREE_B200_H
#define SPAMTREE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct st_handle st_handle; /* opaque: the SpamTreeMV object (src/spamtree_model.h:22-212) */

typedef enum {
  ST_OK = 0,
  ST_ERR_INVALID = 1,   /* bad argument / inconsistent DAG (reference: `throw 1`, spamtree_model.cpp:201-226) */
  ST_ERR_CUDA = 2,      /* CUDA runtime error; st_last_error() has the text */
  ST_ERR_NOT_SPD = 3,   /* Cholesky failed inside the Gibbs step (reference: Rcpp::stop, spamtree_model.cpp:1215-1217) */
  ST_ERR_UNSUPPORTED = 4, /* shape or option outside what this build handles (e.g. mvbias != 0, q > 8) */
  ST_ERR_NAN = 5        /* NaN log-likelihood at the current theta (reference: `throw 1`, spamtree_fit.cpp:234-237) */
} st_status;

/* Multi-GPU: one problem cut into subtrees, one rank (process + GPU) per run of subtrees (SURVEY §8e; the reference is
 * single-process).  Every rank creates its handle from ITS blocks: the blocks of the first n_top_levels tree levels are
 * present on every rank (replicated, computed redundantly), the rest are the rank's own subtrees.  The library calls
 * `allreduce` (in-place sum over ranks of `count` doubles at a DEVICE pointer, after synchronising its stream) for the
 * three scalars of the log-density, the messages of the cut-level blocks to the replicated blocks, and the beta / tausq
 * sufficient statistics.  spamtree_b200/partition.py builds these inputs; the callback is torch.distributed (NCCL). */
typedef int (*st_allreduce_fn)(void* ctx, void* device_ptr, int64_t count);
typedef struct {
  int32_t rank, nranks;
  int32_t n_top_levels;         /* replicated levels (0: the ranks hold disjoint trees) */
  int64_t rng_row_offset;       /* rows owned by lower ranks: keeps the device normal streams of the ranks disjoint */
  int64_t n_global_rows;        /* rows of the whole problem */
  const int64_t* global_rows;   /* n_all, required: row of the whole problem behind every local row (keys the device random
                                   streams; the host stream draws for all rows of the problem on every rank) */
  st_allreduce_fn allreduce;
  void* ctx;
} st_partition;

/* Inputs of the SpamTreeMV constructor (spamtree_model.cpp:8-37), i.e. the arguments
 * spamtree_mv_mcmc receives from R (spamtree_fit.cpp:5-54).  Lists of uvec are CSR.
 * Accepted-and-ignored reference arguments (Z values, blocking, gix_block, start_w,
 * use_alg; SURVEY App. D #6) have no field here. */
typedef struct {
  int64_t n_all;               /* rows incl. rows whose y is missing */
  int32_t p;                   /* covariates */
  int32_t q;                   /* outcomes = #unique(mv_id) */
  const double* y;             /* n_all; NaN = missing (to be predicted) */
  const double* X;             /* n_all x p */
  const double* coords;        /* n_all x 2 */
  const int64_t* mv_id;        /* n_all, 1-based outcome id */
  int32_t n_blocks;
  const int64_t* indexing_ptr; /* n_blocks+1 */
  const int64_t* indexing_idx; /* rows of each block, ascending (R/spamtree_fit.R:324) */
  const int64_t* parents_ptr;  /* n_blocks+1 */
  const int64_t* parents_idx;  /* make_edges output, tree_dep.cpp:113-119 */
  const int64_t* children_ptr; /* n_blocks+1 */
  const int64_t* children_idx; /* make_edges output, tree_dep.cpp:102-110 */
  const double* block_names;   /* n_blocks, 1-based names (layer_names) */
  const double* block_groups;  /* n_blocks, tree level of block id i (layer_gibbs_group) */
  const int64_t* res_is_ref;   /* n_res flags per tree level */
  int32_t n_res;
  int32_t limited_tree;        /* 1: every block conditions on its direct parent only (make_edges_limited, tree_dep.cpp:133-186;
                                  spamtree_model.cpp:901-903, 1275-1278) */
  const double* theta;         /* n_theta start values (covariance_functions.cpp:34-52 layout) */
  int32_t n_theta;
  const double* beta;          /* p start values */
  double tausq;                /* start value (the ctor receives 1/tausq, spamtree_fit.cpp:104) */
  int32_t device;              /* CUDA device ordinal; < 0: host-only handle (bookkeeping for st_get_index, no compute) */
  int32_t keep_H;              /* 1: keep H = w_cond_mean_K of observed blocks and the Sigi_tot / Smu_tot probes of the Gibbs
                                  sweep on the device (needed by st_get_node_state "H", "Sigi_tot", "Smu_tot"); 0: production */
  int64_t smem_panel_bytes;    /* 0 = default; shared-memory budget for one BUILD work group */
  const st_partition* partition; /* NULL: the whole problem on one GPU */
} st_problem;

/* SpamTreeMV::SpamTreeMV — spamtree_model.cpp:8-192 (+ init_indexing :315, na_study :303,
 * make_gibbs_groups :194, init_finalize :355, init_model_data :422).  Copies inputs. */
int st_create(const st_problem* prob, st_handle** out);
void st_destroy(st_handle* h);
/* text of the last error on this handle (or of the last failed st_create when h == NULL) */
const char* st_last_error(const st_handle* h);

/* slot: 0 = param_data, 1 = alter_data (tree_utils.h:63-102; spamtree_model.h:112-113) */

/* SpamTreeMV::theta_update — spamtree_model.cpp:1420-1422 */
int st_theta_update(st_handle* h, int slot, const double* theta);
/* SpamTreeMV::get_loglik_comps_w — spamtree_model.cpp:829-998 (BUILD).
 * out3 = {loglik_w, logdetCi, ok}; ok == 0 (some Cholesky failed) is NOT an error:
 * the reference returns false and the proposal is rejected (spamtree_fit.cpp:223,249). */
int st_get_loglik_comps_w(st_handle* h, int slot, double* out3);
/* SpamTreeMV::deal_with_w(true) — spamtree_model.cpp:1000-1226 (GIBBS sweep over w).
 * z: n_all standard normals in boundary order (the reference's bigrnorm, :1018), or NULL to
 * draw them on the device from (seed, counter). */
int st_deal_with_w(st_handle* h, const double* z, uint64_t seed);
/* SpamTreeMV::get_loglik_w — spamtree_model.cpp:776-826 (LLW). out2 = {loglik_w, logdetCi} */
int st_get_loglik_w(st_handle* h, int slot, double* out2);
/* SpamTreeMV::accept_make_change — spamtree_model.cpp:1432-1435 */
int st_accept_make_change(st_handle* h);
/* SpamTreeMV::predict(theta_changed) — spamtree_model.cpp:1229-1358; uses the z of the last st_deal_with_w */
int st_predict(st_handle* h, int theta_changed);
/* SpamTreeMV::gibbs_sample_beta — spamtree_model.cpp:1364-1391. zb: p*q normals or NULL (host stream).
 * faithful_index != 0 reproduces the reference's row mis-indexing with missing data (SURVEY App. D #12). */
int st_gibbs_sample_beta(st_handle* h, const double* zb, int faithful_index);
/* SpamTreeMV::gibbs_sample_tausq — spamtree_model.cpp:1393-1417. fixed: q values to set tausq_inv to, or NULL to draw */
int st_gibbs_sample_tausq(st_handle* h, const double* fixed);
/* seed of the host random stream used by the two functions above and by st_mcmc_run */
int st_seed(st_handle* h, uint64_t seed);

/* public fields the driver reads/writes (spamtree_fit.cpp:118-120, 378-384) */
int st_get_w(st_handle* h, double* w_out /* n_all, boundary order */);
int st_set_w(st_handle* h, const double* w_in);
int st_get_params(st_handle* h, double* Bcoeff /* p x q or NULL */, double* tausq_inv /* q or NULL */,
                  double* XB /* n_all or NULL */);
int st_set_tausq_inv(st_handle* h, const double* tausq_inv /* q */);

/* Per-block state for parity tests.  which:
 *  "H"  w_cond_mean_K(u)  m x P      (spamtree_model.cpp:887)      [needs keep_H]
 *  "Ri" Rcc_invchol(u)    m x m      (:896) ; for non-reference blocks ccholprecdiag(u), m (:945)
 *  "Sigi_tot" m x m (:1044-1051) and "Smu_tot" m (:1062-1077) as seen by the last st_deal_with_w
 *             (non-reference blocks: m scalars each, :1123-1127)
 *  "logdetCi_comps" / "loglik_w_comps": all blocks (u ignored), n_blocks values (:966-968)
 * Writes at most cap doubles; *count receives the element count. */
int st_get_node_state(st_handle* h, int slot, int u, const char* which, double* out, int64_t cap, int64_t* count);

/* Integer bookkeeping for bit-exact parity (spamtree_model.cpp:194-420).  which:
 *  "parents_indexing" (u) · "dim_by_parent" (u) · "this_is_jth_child" (u) · "u_by_block_groups" (u = group)
 *  "blocks_not_empty" · "blocks_predicting" · "block_is_reference" · "block_ct_obs" · "n_actual_groups"
 *  "u_is_which_col" (u, c = child position): {firstcol, lastcol} of spamtree_model.cpp:395-396 */
int st_get_index(st_handle* h, const char* which, int u, int c, int64_t* out, int64_t cap, int64_t* count);

/* ---- the MCMC driver: spamtree_mv_mcmc, spamtree_fit.cpp:5-430 ---- */
typedef struct {
  const double* set_unif_bounds; /* npar x 2 */
  const double* mcmcsd;          /* npar x npar */
  int32_t keep, burn, thin;
  int32_t adapting, sample_beta, sample_tausq, sample_theta, sample_w, sample_predicts;
  int32_t faithful_beta_index;   /* see st_gibbs_sample_beta */
  int32_t rng_mode;              /* 0: host-driven chain, every draw from one host stream in the reference's order (lock-step with
                                    the oracle and with the reference's own driver; one host round trip per step);
                                    1: device-resident chain: proposal, accept decision, slot swap, RAM adaptation, tausq / beta
                                    draws and yhat on the device from Philox streams keyed by (seed, row or parameter,
                                    iteration); the host only enqueues and synchronises once, at the end of the run */
  uint64_t seed;
} st_mcmc_opts;
typedef struct {                 /* caller-allocated; NULL pointers are skipped */
  double* beta_mcmc;             /* p x keep x q */
  double* tausq_mcmc;            /* q x keep */
  double* theta_mcmc;            /* npar x keep */
  double* w_mcmc;                /* n_all x keep */
  double* yhat_mcmc;             /* n_all x keep */
  double* paramsd;               /* npar x npar */
  double mcmc_time;              /* seconds, like the reference's return value (spamtree_fit.cpp:394,413) */
  int64_t n_accepted, n_chol_fail;
} st_mcmc_out;
int st_mcmc_run(st_handle* h, const st_mcmc_opts* opts, st_mcmc_out* out);

/* ---- prediction at new locations from saved samples (no reference counterpart; the math is predict_std,
 * spamtree_model.cpp:1234-1358, and the yhat of spamtree_fit.cpp:384, per saved sample s):
 *   w_new,i = K_{i,pa} K_pa^-1 w_pa,s + sqrt(K_ii - K_{i,pa} K_pa^-1 K_{pa,i}) z_i     (covariance at theta_s; sd 0 when
 *                                                                                      the Schur complement is not positive)
 *   y_new,i = x_i' beta_s[:, mv_i] + w_new,i + sqrt(tausq_s[mv_i]) eps_i
 * pa = the parent list of the row's group (st_tree_attach).  The handle's fitted state is not changed: the current slot,
 * w, beta, tausq and the chain state stay as they are; the alter slot is used as scratch for the BUILD of each distinct
 * theta_s: until st_get_loglik_comps_w(h, 1, ...) or st_mcmc_run rebuilds it, st_accept_make_change and
 * st_get_loglik_w(h, 1, ...) return ST_ERR_INVALID.  Samples that repeat the previous theta bit for bit skip that BUILD.
 * ST_ERR_NOT_SPD: the covariance at some sample's theta is not positive definite on a reference block (a chain never saves
 * such a theta); the outputs are then not draws of the model.  Single-GPU handles only (ST_ERR_UNSUPPORTED otherwise). */
typedef struct {
  int64_t n_new;
  const double* coords;        /* n_new x 2 */
  const int64_t* mv_id;        /* n_new, 1-based */
  const double* X;             /* n_new x p, or NULL: no covariates (x' beta = 0) */
  int64_t n_groups;
  const int64_t* group;        /* n_new: 0-based group of each row */
  const int64_t* parents_ptr;  /* n_groups + 1 */
  const int64_t* parents_idx;  /* 0-based block ids of each group's parents, root first (a chain of reference blocks, as
                                  st_tree_attach returns; limited trees: the direct parent only) */
} st_new_rows;
typedef struct {
  int32_t n_samples;           /* S */
  const double* theta;         /* npar x S */
  const double* beta;          /* p x S x q (beta_mcmc's layout) */
  const double* tausq;         /* q x S */
  const double* w;             /* n_all rows per sample, boundary order: w(i, s) = w[i * w_row_stride + s * w_sample_stride];
                                  one of the two strides must be 1 (st_mcmc_out.w_mcmc: 1, n_all; its C-order transpose: S, 1) */
  int64_t w_row_stride, w_sample_stride;
  const double* z;             /* n_new x S normals of the w draws, or NULL: drawn on the device */
  const double* eps;           /* n_new x S normals of the y draws, or NULL */
  uint64_t seed;               /* device draws: Philox keyed by (seed, new row, position of the sample in this call) */
} st_pred_samples;
typedef struct {               /* caller-allocated, NULL pointers are skipped; rows in the caller's order */
  double* w_new;               /* n_new x S */
  double* y_new;               /* n_new x S */
  double* mean;                /* n_new x S: K_{i,pa} K_pa^-1 w_pa,s */
  double* sd;                  /* n_new x S: the conditional sd */
  double* w_mean;              /* n_new: mean over the S draws */
  double* w_sd;                /* n_new: sd over the S draws (ddof = 1; 0 for one sample) */
  double* y_mean;              /* n_new */
  double* y_sd;                /* n_new */
  int64_t n_builds;            /* BUILDs of the reference levels run (one per change of theta along the samples) */
} st_pred_out;
int st_predict_new(st_handle* h, const st_new_rows* rows, const st_pred_samples* samples, st_pred_out* out);

/* ---- draws kept on the device and summarised there (no reference counterpart; DESIGN.md §5c) ----
 * st_keep_samples_on_device: for the following st_mcmc_run calls with rng_mode = 1, keep the saved iterations' w and / or
 * yhat in device memory, [sample][row] (one contiguous n_all vector per saved iteration, boundary order).  Host copies are
 * still made where st_mcmc_out.w_mcmc / yhat_mcmc are not NULL, and the chain draws exactly what it draws without the store.
 * The store (n_all x keep x 8 bytes per quantity) is checked against the free device memory before a run allocates or
 * launches anything: ST_ERR_UNSUPPORTED, with the bytes needed and free, and the handle as it was.  It holds the last completed
 * run, is replaced by the next one, and is freed by what = 0 or st_destroy.  ST_ERR_UNSUPPORTED: a store with rng_mode = 0,
 * or on a partitioned handle.
 * ST_KEEP_LOGLIK_INT: the integrated log-likelihood of every row at every saved iteration (DESIGN.md §5f), [sample][row] in
 * boundary order, NaN at the rows whose y is missing.  Row i of draw s is ll = log N(y_i - x_i' beta; m_i, v_i + tausq_j), where
 * N(m_i, v_i) is the prior conditional of w_i given the rest of w at theta_s, as the Gibbs sweep has it when it draws the block
 * of row i, and beta, tausq are those the sweep uses.  Only the saved iterations' sweeps form it (with the same draws: the chain
 * is bit for bit the chain without it).  Refused with ST_ERR_INVALID by an st_mcmc_run that does not sample w, besides the
 * refusals above; st_deal_with_w forms it too while the bit is set (st_get_loglik_int). */
#define ST_KEEP_W 1
#define ST_KEEP_YHAT 2
#define ST_KEEP_LOGLIK_INT 4
int st_keep_samples_on_device(st_handle* h, int32_t what);
/* The integrated log-likelihood of the last sweep that formed it (st_deal_with_w with ST_KEEP_LOGLIK_INT set, or the last saved
 * iteration of an st_mcmc_run with it), n_all values in boundary order, NaN where y is missing.  ST_ERR_INVALID: no sweep has
 * formed it on this handle. */
int st_get_loglik_int(st_handle* h, double* out);
/* Copies the draws of a device store to the host: which as st_summarize, and 4 = the integrated log-likelihood of the last
 * stored run.  out: n_rows x n_samples doubles, [sample][row] (out NULL: the sizes only).  ST_ERR_INVALID: nothing stored. */
int st_copy_store(st_handle* h, int32_t which, double* out, int64_t* n_rows, int32_t* n_samples);
/* Per-row summaries of stored draws.  which: 0 = w, 1 = yhat of the last stored run (rows in boundary order); 2 = w_new,
 * 3 = y_new of the last st_predict_new_stored with keep_draws (rows in the caller's order).  Over the S draws of a row:
 *   mean; sd (ddof = 1, 0 for S = 1); quantiles at probs[0..n_probs) exactly as numpy.quantile(method="linear") (R type 7);
 *   batch means with b = floor(sqrt(S)) draws per batch over the first B = floor(S / b) batches: sigma2 = b var(batch means,
 *   ddof = 1), mcse = sqrt(sigma2 / S), ess = S var(draws, ddof = 1) / sigma2, both NaN when S < 2 or sigma2 = 0.
 * Every reduction runs in a fixed order: repeated calls are bit-identical.  ST_ERR_INVALID: nothing stored for `which`, or a
 * prob outside [0, 1] or NaN; ST_ERR_UNSUPPORTED: S above what one CTA can stage (the limit is in the message). */
typedef struct {               /* caller-allocated; NULL pointers are skipped (all NULL: only the sizes are returned) */
  double* mean;                /* n_rows */
  double* sd;                  /* n_rows */
  double* quantiles;           /* n_rows x n_probs */
  double* mcse;                /* n_rows */
  double* ess;                 /* n_rows */
  int64_t n_rows;              /* out */
  int32_t n_samples;           /* out */
} st_summary_out;
int st_summarize(st_handle* h, int32_t which, const double* probs, int32_t n_probs, st_summary_out* out);
/* st_predict_new from every saved iteration of the last stored run (ST_KEEP_W required, else ST_ERR_INVALID): theta, beta and
 * tausq of the run, w_s read from the device store; normals from the device (seed as st_pred_samples.seed).  The outputs are
 * those st_predict_new gives for the same samples as host arrays.  keep_draws != 0: the w_new / y_new draws also go to a device
 * store (n_new x S each, [sample][row], checked against the free memory like the run's) for st_summarize(which = 2, 3). */
int st_predict_new_stored(st_handle* h, const st_new_rows* rows, uint64_t seed, int32_t keep_draws, st_pred_out* out);

/* ---- several chains: pooled summaries and convergence diagnostics (no reference counterpart; DESIGN.md §5d) ----
 * K chains of S draws per row.  Over all K S draws of a row, pooled: mean; sd (ddof = 1, 0 for one draw); quantiles at
 * probs[0..n_probs) exactly as numpy.quantile(method="linear").  Per row, as ArviZ's rhat(method="rank") and
 * ess(method="bulk" | "tail") define them (Vehtari, Gelman, Simpson, Carpenter and Buerkner 2021), with h = S / 2:
 *   split: each chain gives its first h and its last h draws, M = 2K chains of h (odd S: the middle draw is in no split chain,
 *   but is in the pooled statistics and the tail thresholds); z-scale: Phi^-1((r - 3/8) / (M h + 1/4)) of the average ranks
 *   r (ties averaged) of the M h split draws;
 *   rhat = max(R(z-scale(split x)), R(z-scale(|split x - median(split x)|))), R(y) = sqrt((B / W + h - 1) / h) with B = h
 *   var(chain means, ddof 1), W = mean of the within-chain variances (ddof 1); NaN if either R is (W = 0);
 *   ess_bulk = ESS(z-scale(split x)); ess_tail = min(ESS(split 1[x <= q05]), ESS(split 1[x <= q95])), q05 / q95 the pooled
 *   0.05 / 0.95 quantiles, NaN if either is; ESS: Geyer's initial positive and monotone sequences over the mean biased
 *   autocovariances, tau >= 1 / log10(M h), NaN when the pooled variance estimate is 0;
 *   rhat, ess_bulk and ess_tail are NaN for S < 4 (h < 2).
 * Draws must be finite: a chain's stored draws are (a run with a NaN log-likelihood stops with ST_ERR_NAN), and
 * st_summarize_draws refuses non-finite host draws (ST_ERR_INVALID, with the index of the first).
 * Every reduction runs in a fixed order: repeated calls are bit-identical.  Refused: n_chains < 1, n_samples < 1, a prob
 * outside [0, 1] or NaN (ST_ERR_INVALID); n_chains x (n_samples + 1) above what one CTA stages in shared memory
 * (ST_ERR_UNSUPPORTED, the limit in the message). */
typedef struct {            /* caller-allocated; NULL pointers are skipped (all NULL: only the sizes are returned) */
  double* mean;             /* n_rows */
  double* sd;               /* n_rows */
  double* quantiles;        /* n_rows x n_probs (column-major) */
  double* rhat;             /* n_rows */
  double* ess_bulk;         /* n_rows */
  double* ess_tail;         /* n_rows */
  int64_t n_rows;           /* out */
  int32_t n_chains, n_samples;  /* out */
} st_chains_summary_out;
/* The device stores of `which` (as st_summarize: 0 = w, 1 = yhat, 2 = w_new, 3 = y_new) on n_chains handles, read in place.
 * Every handle must be on the same device and store the same n_rows and S, else ST_ERR_INVALID naming the first handle that
 * differs; a handle with nothing stored for `which` gives ST_ERR_INVALID.  That the handles were built from the same problem
 * (so that row i means the same location on each) is the caller's responsibility.  Waits for every handle's stream, runs on
 * that of hs[0] and returns when done; changes no handle's state (store, chain, slots, st_keep_samples_on_device mask).
 * Errors: st_last_error(hs[0]); st_last_error(NULL) when there is no handle to report to (hs or hs[0] NULL, n_chains < 1). */
int st_summarize_chains(st_handle* const* hs, int32_t n_chains, int32_t which, const double* probs, int32_t n_probs,
                        st_chains_summary_out* out);
/* The same on host draws [chain][sample][row] (n_chains x n_samples x n_rows), copied to `device` for the call and freed after
 * it: ST_ERR_UNSUPPORTED when the copy does not fit in the free device memory.  No handle: errors are st_last_error(NULL). */
int st_summarize_draws(int32_t device, const double* draws, int64_t n_rows, int32_t n_chains, int32_t n_samples,
                       const double* probs, int32_t n_probs, st_chains_summary_out* out);

/* ---- model criteria: PSIS-LOO with Pareto k-hat, WAIC and DIC per observation (no reference counterpart; DESIGN.md §5e) ----
 * K chains x S saved iterations, N = K S pooled draws g = c S + s.  For an observed row i (finite y_i; rows in boundary order,
 * as w_mcmc) with outcome j = mv_id_i, the log-likelihood conditional on w:
 *   ll[i,g] = -0.5 log(2 pi tausq[j,g]) - (y_i - x_i' beta[:,j,g] - w[i,g])^2 / (2 tausq[j,g])
 * (beta p x S x q and tausq q x S as st_mcmc_out holds them; tausq is tau^2).  Rows with a missing y are NaN in every per-row
 * output and are left out of every total; n_obs counts the observed rows.  Per row, LSE = log-sum-exp:
 *   lpd = LSE_g(ll) - log N;  p_waic = var_g(ll) (ddof 1, NaN for N = 1);  elpd_waic = lpd - p_waic   (R loo::waic)
 *   PSIS-LOO (R loo 2.x psis(), gpdfit with wip = TRUE, min_grid_pts = 30, prior 3): lw = r - max(r) with r = -ll;
 *   L = tail_len = min(ceil(0.2 N), ceil(3 sqrt(N / r_eff))), k-hat = +Inf; if L >= 5 the largest L sorted lw form the tail
 *   and the sorted value before them the cutoff; unless the tail is constant (max - min < DBL_EPSILON / 100), a generalised
 *   Pareto distribution is fitted to x = exp(tail) - exp(cutoff) (Zhang and Stephens 2009, M = 30 + floor(sqrt(L)) grid
 *   points, k-hat = (L k + 5) / (L + 10), NaN becomes +Inf), and for finite k-hat the tail is replaced by
 *   log(sigma expm1(-k-hat log1p(-p_m)) / k-hat + exp(cutoff)), p_m = (m - 0.5) / L; lw is truncated at 0 and normalised;
 *   elpd_loo = LSE_g(lw + ll), p_loo = lpd - elpd_loo.
 *   DIC (Spiegelhalter et al. 2002, plug-in at the pooled posterior means as spBayes' spDiag): dbar = sum_i -2 mean_g ll,
 *   dhat = sum_i -2 log N(y_i; x_i' mean(beta[:,j]) + mean(w_i), mean(tausq_j)), p_dic = dbar - dhat, dic = dbar + p_dic.
 * Totals over the observed rows: elpd_loo_total = sum, se_elpd_loo = sqrt(n_obs var(elpd_loo_i, ddof 1)), looic = -2
 * elpd_loo_total, se_looic = 2 se_elpd_loo; the same for WAIC; lpd_total; k_threshold = min(1 - 1 / log10(N), 0.7);
 * n_k_high = rows with k-hat > k_threshold (+Inf included); n_p_waic_high = rows with p_waic > 0.4.
 * The criteria condition on w, one latent value per observation, so w_i is informed mostly by y_i itself and PSIS-LOO of such
 * a model often shows k-hat > 0.7 on many rows (Vehtari, Mononen, Tolvanen, Sivula and Winther 2016): n_k_high says how far
 * elpd_loo can be trusted.  Every reduction runs in a fixed order: repeated calls are bit-identical.
 * Refused: r_eff <= 0 or not finite, n_chains < 1, n_samples < 1 (ST_ERR_INVALID); N above what one CTA stages in shared
 * memory (ST_ERR_UNSUPPORTED, the limit in the message). */
typedef struct {                 /* caller-allocated; NULL pointers skipped; all NULL: only the sizes (n_rows, n_obs, n_chains,
                                    n_samples, k_threshold) are returned and the other totals are NaN */
  double *lpd, *elpd_loo, *p_loo, *pareto_k, *elpd_waic, *p_waic;   /* n_rows each, NaN at unobserved rows */
  double elpd_loo_total, se_elpd_loo, p_loo_total, looic, se_looic;  /* out */
  double elpd_waic_total, se_elpd_waic, p_waic_total, waic, se_waic, lpd_total;
  double dbar, dhat, p_dic, dic, k_threshold;
  int64_t n_rows, n_obs, n_k_high, n_p_waic_high;                    /* out */
  int32_t n_chains, n_samples;                                      /* out */
} st_fit_criteria_out;
/* The w stores of n_chains handles read in place, with the beta / tausq samples of the same stored runs and the handles' y,
 * X and mv_id.  Every handle must be on the same device, store the same n_rows and S, and have the same p, q, y, X and mv_id,
 * else ST_ERR_INVALID naming the first handle that differs; a handle without a w store gives ST_ERR_INVALID.  Waits for every
 * handle's stream, runs on that of hs[0] and returns when done; changes no handle's state.  Errors: st_last_error(hs[0]);
 * st_last_error(NULL) when there is no handle to report to. */
int st_fit_criteria(st_handle* const* hs, int32_t n_chains, double r_eff, st_fit_criteria_out* out);
/* Integrated PSIS-LOO and WAIC (DESIGN.md §5f): the same outputs and handle checks as st_fit_criteria, from the stores of the
 * integrated log-likelihood (ST_KEEP_LOGLIK_INT) read in place instead of the log-likelihood conditional on w.  w_i is
 * integrated out of each row's term, so the importance ratios of PSIS-LOO have lighter tails.  The DIC fields are NaN.  A
 * handle without that store gives ST_ERR_INVALID. */
int st_fit_criteria_integrated(st_handle* const* hs, int32_t n_chains, double r_eff, st_fit_criteria_out* out);
/* The PSIS / WAIC part on a host log-likelihood [chain][sample][row] (n_chains x n_samples x n_rows), copied to `device` for
 * the call: a row of NaN is an unobserved row; any other non-finite value is refused (ST_ERR_INVALID).  The DIC fields are NaN
 * (no parameters are given).  ST_ERR_UNSUPPORTED when the copy does not fit in the free device memory.  Errors:
 * st_last_error(NULL). */
int st_fit_criteria_loglik(int32_t device, const double* loglik, int64_t n_rows, int32_t n_chains, int32_t n_samples,
                           double r_eff, st_fit_criteria_out* out);

/* ---- the Metropolis-Hastings glue (mh_adapt.h / mh_adapt.cpp), as st_mcmc_run uses it; host-only, no handle ---- */
/* par_huvtransf_fwd / par_huvtransf_back (Rcpp exports), mh_adapt.cpp:3-15: logit / logistic on (bounds[j], bounds[j + npar]).
 * bounds: npar x 2. */
int st_par_huvtransf_fwd(const double* par, int32_t npar, const double* bounds, double* out);
int st_par_huvtransf_back(const double* par, int32_t npar, const double* bounds, double* out);
/* One proposal as spamtree_fit.cpp:211-215 forms it: new_param = back(fwd(param) + paramsd U), clipped by unif_bounds
 * (mh_adapt.h:188-202).  out: new_param (npar), calc_jacobian(new_param, param) (mh_adapt.h:230-239), out_unif_bounds (0/1). */
int st_mh_propose(int32_t npar, const double* param, const double* bounds, const double* paramsd, const double* U,
                  double* out /* npar + 2 */);
/* do_I_accept, mh_adapt.h:20-36, with the caller's uniform draw u: returns 1 (accept) or 0 */
int st_do_i_accept(double logaccept, double u);
/* class RAMAdapt, mh_adapt.h:40-135, over a recorded sequence: U npar x steps, alpha[steps], iteration numbers 0..steps-1.
 * paramsd_out npar x npar after the last step; paramsd_trace (or NULL) npar*npar per step.  ST_ERR_INVALID when
 * metropolis_sd is not positive definite (arma::chol throws in the reference, :86). */
int st_ram_adapt(int32_t npar, const double* metropolis_sd, int32_t steps, const double* U, const double* alpha,
                 double* paramsd_out, double* paramsd_trace);

/* ---- multi-GPU: native collectives (no reference counterpart) ---- */
/* Native collective path of a partitioned handle: the library owns an NCCL communicator and enqueues its all-reduces
 * on the handle's own stream (no host synchronisation, no callback).  Rank 0 calls st_nccl_unique_id, the 128 bytes
 * are handed to every rank by whatever means the host has (torch.distributed broadcast in spamtree_b200/dist.py), and
 * every rank calls st_attach_nccl on its handle — collectively, like ncclCommInitRank.  libnccl.so.2 is resolved at
 * run time (dlopen), so handles that never attach need no NCCL at all.  Without it the `allreduce` callback is used. */
#define ST_NCCL_UNIQUE_ID_BYTES 128
int st_nccl_unique_id(unsigned char* out128);
int st_attach_nccl(st_handle* h, const unsigned char* id128);

/* ---- bench / profiling hooks (no reference counterpart) ---- */
/* One hot-path iteration without host random draws: GIBBS (device normals) + LLW + BUILD(alter, theta_prop)
 * + optional swap + tausq + beta (spamtree_fit.cpp:167-330 minus predict/save).  ms_out[0..5] (when non-NULL) receive the
 * CUDA-event times of {gibbs (+ Gram refresh), llw, build on the main stream (+ deferred half), tausq + beta, the whole
 * iteration, the upper levels of BUILD on the second stream (0 when the iteration is sequential: then [0..3] add up to [4])}. */
int st_bench_iteration(st_handle* h, const double* theta_prop, int do_swap, uint64_t seed, double* out3, float* ms_out);
/* row index of the beta step used by st_bench_iteration: 1 = the reference's (SURVEY App. D #12, the default on a single-GPU
 * handle), 0 = the corrected one (the only one a partitioned handle supports) */
int st_set_beta_index(st_handle* h, int faithful);
/* counts of kernel launches and algorithmic work: out[8] = {kernel launches since creation, F_alg flops of one iteration
 * (SURVEY §8d formula on the actual tree), executed-flop estimate of the lean formulation, covariance evaluations,
 * F_alg of BUILD alone (F_build), executed-flop estimate of BUILD alone, compulsory output bytes of one BUILD,
 * bytes of the chain state that a device-resident run sends up / brings back once} */
int st_get_counters(st_handle* h, double* out8);
int st_sync(st_handle* h);

/* ---- DAG construction: tree_dep.cpp ---- */
/* kthresholds, tree_dep.cpp:16-27.  res: k-1 values */
int st_kthresholds(const double* x, int64_t n, int32_t k, double* res);
/* part_axis_parallel_lmt, tree_dep.cpp:58-67 (thresholds of axis j at thr[thr_ptr[j]..thr_ptr[j+1])); out n x d */
int st_part_axis_parallel_lmt(const double* coords, int64_t n, int32_t d, const double* thr, const int64_t* thr_ptr,
                              double* out);
/* number_revalue, tree_dep.cpp:240-259 */
int st_number_revalue(const int64_t* orig, int64_t nr, int32_t nc, const int64_t* from_val, const int64_t* to_val,
                      int64_t nfrom, int64_t* out);
/* make_edges / make_edges_limited, tree_dep.cpp:75-186.  parchimat nr x L (NaN = NA, 1-based block names).
 * Two-call protocol: with par_idx == NULL only counts[0..2] = {n_blocks, #parent entries, #child entries} are written. */
int st_make_edges(const double* parchimat, int64_t nr, int32_t L, const int64_t* non_empty_blocks, int64_t n_ne,
                  const int64_t* res_is_ref, int32_t limited, int64_t* par_ptr, int64_t* par_idx, int64_t* chi_ptr,
                  int64_t* chi_idx, int64_t* counts);

/* Deterministic stand-in for R's make_tree() (R/make_tree.R:1-420; SURVEY App. G): same structure, with the
 * per-cell `sample()` (R/make_tree.R:92) replaced by "smallest splitmix64(ix ^ seed) in the cell" and the FNN
 * kd-tree 1-NN replaced by an exact 1-NN.  Rows must already be sorted by (Var1, Var2, ix) as spamtree() does
 * (R/spamtree_fit.R:214).  tree_depth <= 0 means Inf.  Results are fetched from the returned object. */
typedef struct st_tree st_tree;
typedef struct {
  int64_t n_all;
  const double* coords;   /* n_all x 2, sorted */
  const double* y;        /* NaN = missing */
  const int64_t* mv_id;   /* 1-based */
  int32_t cell_size;      /* 25 */
  int32_t K[2];           /* 2,2 */
  int32_t start_level, tree_depth;
  int32_t last_not_reference, cherrypick_same_margin, cherrypick_group_locations;
  uint64_t seed;
} st_tree_opts;
int st_make_tree(const st_tree_opts* o, st_tree** out);
void st_tree_destroy(st_tree* t);
/* sizes: {n_blocks, n_res, parchi rows, parchi cols, #parent entries, #child entries} */
int st_tree_sizes(const st_tree* t, int64_t* out6);
/* blocking/res: n_all (1-based block name and tree level of each row); parchimat: rows x cols (NaN = NA);
 * the rest is exactly what st_problem takes.  Any pointer may be NULL. */
int st_tree_get(const st_tree* t, int64_t* blocking, int64_t* res, int64_t* res_is_ref, double* parchimat,
                int64_t* indexing_ptr, int64_t* indexing_idx, int64_t* parents_ptr, int64_t* parents_idx,
                int64_t* children_ptr, int64_t* children_idx, double* block_names, double* block_groups);
/* New rows attached to a built tree (no reference counterpart; the rule is that of the prediction level, R/make_tree.R:317-413):
 * the nearest row of the last loop level (same margin first when the tree was built with cherrypick_same_margin) names the
 * parent block b; the new rows of one b form one group, groups numbered by ascending b; a group's parents are the reference
 * blocks on the chains through b, root first (make_edges' rule for a column appended to parchimat; limited != 0: the last of
 * them, make_edges_limited).  The tree itself is not changed.  coords_new n_new x 2, mv_new 1-based.
 * group: n_new (0-based group of each row); par_ptr: n_groups + 1; par_idx: 0-based block ids.
 * Two-call protocol: with par_idx == NULL only counts[0..1] = {n_groups, #parent entries} are written. */
int st_tree_attach(const st_tree* t, int64_t n_new, const double* coords_new, const int64_t* mv_new, int32_t limited,
                   int64_t* group, int64_t* par_ptr, int64_t* par_idx, int64_t* counts);

/* CrossCovarianceAG10 (R export), covariance_functions.cpp:301-355, evaluated on the GPU.
 * coords n x 2 col-major, mv 1-based, Dmat q x q; out n1 x n2. */
int st_cross_covariance_ag10(const double* coords1, const int64_t* mv1, int64_t n1, const double* coords2,
                             const int64_t* mv2, int64_t n2, const double* ai1, const double* ai2,
                             const double* phi_i, const double* thetamv, int32_t n_thetamv, const double* Dmat,
                             int32_t q, int32_t device, double* out);

/* library info: returns a static string "spamtree_b200 <version> sm_100a" */
const char* st_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SPAMTREE_B200_H */
