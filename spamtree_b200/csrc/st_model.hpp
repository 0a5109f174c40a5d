// st_model.hpp — host mirror of the reference's SpamTreeMV (src/spamtree_model.h:22-212) with its state on one GPU.
//
// Layout decisions (DESIGN.md §3):
//  * rows are permuted ONCE into node-major order (level, node, row) so that a block's rows and each ancestor panel are
//    contiguous; outputs are un-permuted only at the boundary (st_get_w);
//  * per block and per theta-slot only G = Ri*H (m x P), Ri (m x m) and (optionally) H are kept — the reference's Kxc,
//    Kxx_inv, Kxx_invchol, AK_uP_all, AK_uP_u_all and Sigi_children cubes are never materialised (SURVEY App. F);
//  * a block's parent set is its ancestor chain (tree_dep.cpp:113-119); G is stored as the block's rows of the chain's
//    inverse Cholesky factor, [ G | -Ri | 0 ] row-major, so that BUILD of the descendants streams contiguous rows.
#pragma once
#include <cuda_runtime.h>

#include <functional>
#include <initializer_list>
#include <string>
#include <vector>

#include "../../include/spamtree_b200.h"
#include "st_chain.hpp"
#include "st_common.hpp"

namespace st {

bool make_covtab(const double* theta, int n_theta, int q, CovTab& tab, std::string& err);

// device pointers describing the tree (read-only after st_create)
struct DevTree {
  // per row, node-major
  const double* cx;
  const double* cy;
  const int* mvq;        // 0-based outcome
  const double* y;       // missing -> 0 (spamtree_model.cpp:146)
  const double* X;       // n_all x p column-major, node-major rows
  // per node (slot)
  const int* m;
  const int* row0;
  const int* isref;      // 1: reference level (full m x m conditional), 0: rows conditionally independent
  const int* k;          // chain length (#reference ancestors)
  const int* P;          // parent-set size
  const int* lastpar;    // slot of the last (deepest) parent, -1 for roots
  const int* chain_off;  // into the per-chain-entry arrays
  const long long* goff; // G / H storage offset (doubles) of the block's row block
  const int* gs;         // row stride of that row block: [ G (P) | -Ri (m, reference blocks) | 0 ], g_stride()
  const long long* moff; // limited trees: offset (in the G array) of the block's MARGINAL factor rows [ -chol(K_uu)^-1 | 0 ], stride (m+3)&~3; -1: none
  int limited;           // 1: limited tree (children stream the parent's marginal factor, spamtree_model.cpp:901-903)
  const long long* rioff;// Ri storage offset (doubles)
  const long long* voff; // message vector offset (P doubles)
  const long long* uoff; // message Gram offset (tiles m_a x m_a per ancestor); unused when ufused
  const int* ufused;     // 1: childless block whose Gram tiles are formed by its parent on the fly (never stored)
  const long long* soff; // child-sum Gram (m x m) offset, -1 when the node has no children
  const int* child_ptr;
  const int* child_idx;  // direct observed children (slots)
  // per chain entry
  const int* chain;      // ancestor slot, root first
  const int* chain_poff; // column offset of the ancestor inside the parent set
  const int* chain_uoff; // offset (doubles) of the ancestor's tile inside the node's Gram storage
};

struct DevSlot {  // everything that depends on theta (tree_utils.h:63-102, lean form)
  double* G;
  double* H;       // nullptr when keep_H == 0 (prediction blocks always keep theirs in Hpred)
  double* Ri;
  double* logdet;  // per node
  double* llcomp;  // per node
};

// both theta-slots plus the chain state that says which one is param_data: kernels pick their slot on the device, so an
// accepted proposal (accept_make_change) needs no host involvement
struct DevSlots {
  DevSlot s[2];
  const ChainDev* chain;
};

struct LevelInfo {
  int slot0 = 0, nslots = 0;  // node range
  int is_ref = 1;
  int grp0 = 0, ngrp = 0;     // BUILD work groups (index into grp arrays)
  // the groups of a level are bucketed by width (8-column tiles) so that narrow groups are not launched with the
  // shared memory and CTA size of the widest one
  struct BuildLaunch {
    int grp0 = 0, ngrp = 0;
    size_t smem = 0;          // dynamic shared memory of build_level_kernel
    int threads = 128;        // 32 x (8-column tiles of the widest group in the bucket), at least 4 warps
    int ns = 2;               // depth of the cp.async ring (1 when that lets two CTAs share an SM, or when 2 does not fit)
  };
  std::vector<BuildLaunch> build_launches;
  // childless non-reference level: BUILD runs its forward half only (log-density) and parks Z in G's storage; the
  // backward half runs when the slot is taken up (accepted proposal).  Not when H is kept (parity getters).
  bool deferrable = false;
  int maxP = 0, maxm = 0, maxNC = 0, maxk = 0;
  size_t smem_gibbs = 0;
  int gram_rch = 1, gram_ldx = 2, gram_tiles = 2, gram_stage_off = 2, gram_threads = 256;  // gram_level_kernel: staged rows per chunk, their leading dimension, doubles of the assembled tiles
  bool gram_skip = false;          // every block of the level is fused into its parent
  int gram_maxrows = 0, gram_maxitems = 0;  // largest rows a block stages (own + fused children), largest (tile, sub-block) item count
};

struct GroupSpec { int s, nn, NT; };  // a BUILD work group: nn sibling blocks from slot s, NT tiles of 8 columns

// Rows a kernel writes on `stream` go to slices of the caller's host arrays on the copy stream, while the work enqueued
// after them runs (DESIGN.md §5).  One per run or call: open() page-locks the caller's ranges where it can and allocates
// the staging slots, buffer() hands out a slot once the last copy that read it is done (a wait of the stream, not of the
// host), send() issues the copies, finish() waits for all of them.  A range that cannot be page-locked (pageable memory
// the driver refuses, or memory that is page-locked already) takes the same copies: into pageable memory a device-to-host
// copy returns only once it is complete, so only when a copy runs can change, never what arrives.  Status: 0, or
// ST_ERR_CUDA with `err` set.
class CopyOut {
 public:
  CopyOut(cudaStream_t stream, cudaStream_t copy_stream, std::string& err) : st_(stream), cs_(copy_stream), err_(err) {}
  ~CopyOut();  // waits for both streams, unlocks the ranges, frees the staging
  CopyOut(const CopyOut&) = delete;
  CopyOut& operator=(const CopyOut&) = delete;
  // hosts: the caller's arrays (NULL skipped), bytes_each bytes from each; nslots staging slots of n doubles
  int open(std::initializer_list<double*> hosts, size_t bytes_each, int nslots, size_t n);
  double* buffer(int slot);  // NULL on a CUDA error
  // dst[c] <- src[c], n doubles each (NULL dst skipped), once what `stream` holds so far has run; `slot`: the staging slot
  // the sources are in, whose next buffer() waits for these copies
  int send(int slot, double* const* dst, const double* const* src, int count, size_t n);
  int finish();

 private:
  int chk(cudaError_t e, const char* what);
  cudaStream_t st_, cs_;
  std::string& err_;
  std::vector<void*> locked_;
  double* staging_ = nullptr;
  size_t n_ = 0;
  cudaEvent_t ready_ = nullptr;
  std::vector<cudaEvent_t> copied_;  // per slot
  std::vector<char> pending_;
};

// Draws kept on the device (st_keep_samples_on_device, st_predict_new_stored, st_summarize; DESIGN.md §5c), the only code
// that knows the stores' layout.  Store k holds [sample][row] draws, n rows x S samples: w (0), yhat (1) and the integrated
// log-likelihood (4) of the last device-resident run, w_new (2) and y_new (3) of the last stored prediction.  A mask selects
// store k by bit k (mask_of turns an st_keep_samples_on_device mask into one).
class DrawStore {
 public:
  static constexpr int kStores = 5, kLoglikInt = 4;
  static constexpr int kRun = 3 | (1 << kLoglikInt), kPrediction = 12;  // what a run, a stored prediction replaces
  static int mask_of(int keep) { return (keep & (ST_KEEP_W | ST_KEEP_YHAT)) | ((keep & ST_KEEP_LOGLIK_INT) ? 1 << kLoglikInt : 0); }
  struct Store {
    double* d = nullptr;
    size_t cap = 0;  // bytes allocated (reused by the next run when large enough)
    int64_t n = 0;
    int S = 0;       // 0: holds nothing
  };
  DrawStore() = default;
  DrawStore(const DrawStore&) = delete;
  DrawStore& operator=(const DrawStore&) = delete;
  ~DrawStore() { release(); }
  // empties the stores of the groups (kRun, kPrediction) that `mask` touches, makes room for bytes_each bytes in each
  // store of `mask` and frees the group's others.  Refused (ST_ERR_UNSUPPORTED) when that does not fit the free device
  // memory plus what those stores hold already: then every store is as it was
  int reserve(int mask, size_t bytes_each, const char* what, std::string& err);
  void commit(int mask, int64_t n, int S);  // a completed run or prediction wrote S draws of n rows into each store of mask
  const Store& get(int which) const { return s_[which]; }
  // the store, or NULL and err = who + "no stored draws of <name> (<how to keep them>)"
  const Store* find(int which, const std::string& who, std::string& err) const;
  void release();
  dvec samples;  // theta (npar x S), beta (p x S x q), tausq (q x S) of the last stored run

 private:
  Store s_[kStores];
};

class Model {
 public:
  ~Model();
  // ---- inputs (copied)
  int64_t n_all = 0;
  int p = 0, q = 0, n_blocks = 0;
  dvec y, X, coords;
  ivec mv_id;
  CSR indexing, parents, children;
  dvec block_names, block_groups;
  ivec res_is_ref;
  bool keep_H = true;
  bool limited = false;  // limited_tree (spamtree_model.cpp:67)
  int device = 0;
  size_t smem_budget = 227 * 1024 - 5 * 1024;  // dynamic; the kernel also holds ~4.5 KB of static shared memory (227 KB per CTA)
  int force_build_ns = 0;    // development override of the ring depth (ST_BUILD_NS)
  bool use_pdl = true;       // level launches of a BUILD use programmatic dependent launch (ST_PDL=0 disables)
  bool defer_leaves = true;  // childless non-reference levels: backward half of BUILD only when the slot is taken up (ST_DEFER=0 disables)
  int max_group_cols = 104;  // upper bound on the columns one BUILD work group handles (one warp per 8 columns)
  int n_sm = 148;            // SMs of the device (B200: 148; queried at init when the handle has a device)
  int spread_ctas = -1;      // levels with few blocks use smaller groups, as long as the groups stay within this many CTAs (default: the SM count; ST_SPREAD; 0 disables)
  bool probes = true;        // record Sigi_tot / Smu_tot of the last Gibbs sweep (st_get_node_state)
  // ---- bookkeeping, same meaning as the reference's members
  int64_t n_obs = 0;
  ivec na_ix_all;
  ivec block_ct_obs, blocks_not_empty, blocks_predicting, block_is_reference;
  std::vector<ivec> u_by_block_groups;
  int n_gibbs_groups = 0, n_actual_groups = 0;
  std::vector<SmallMat> XtX;  // per outcome (spamtree_model.cpp:151-155)
  ivec nobs_by_q;
  // ---- node-major layout
  int n_obs_nodes = 0, n_nodes = 0;
  std::vector<int> slot_of_block, block_of_slot;
  std::vector<int> h_m, h_row0, h_k, h_P, h_chain_off, h_chain, h_chain_poff, h_chain_uoff, h_lastpar, h_gs;
  std::vector<long long> h_goff, h_rioff, h_voff, h_uoff, h_soff, h_moff;
  std::vector<int> h_child_ptr, h_child_idx, h_ufused;
  ivec perm;   // node-major row -> boundary row
  ivec iperm;  // boundary row -> node-major row
  std::vector<LevelInfo> levels;  // observed levels, root first
  LevelInfo pred_level;           // prediction blocks
  std::vector<int> h_grp_slot0, h_grp_nn;
  long long g_total = 0, ri_total = 0, v_total = 0, u_total = 0, s_total = 0, gpred_total = 0;
  // ---- multi-GPU partition (include/spamtree_b200.h: st_partition)
  bool part = false;
  int rank = 0, nranks = 1, n_top_levels = 0;
  int64_t rng_row_offset = 0, n_global_rows = 0;
  ivec global_rows;
  int (*allreduce_fn)(void*, void*, int64_t) = nullptr;
  void* allreduce_ctx = nullptr;
  int n_top_slots = 0, n_top_rows = 0, n_slots_total = 0;
  std::vector<int> h_front_pseudo, h_front_c0, h_front_c1, h_front_vlen, h_front_ulen;
  int *d_front_pseudo = nullptr, *d_front_c0 = nullptr, *d_front_c1 = nullptr, *d_front_vlen = nullptr, *d_front_ulen = nullptr;
  long long v_front0 = 0, v_front_len = 0, u_front0 = 0, u_front_len = 0;
  int allreduce_dev(double* dptr, int64_t n);
  // native path: library-owned NCCL communicator, all-reduces enqueued on `stream` (st_attach_nccl)
  void* nccl_comm = nullptr;
  int attach_nccl(const unsigned char* id128);
  int partition_reduce_constants(std::string& e);  // XtX and per-outcome counts summed over the ranks
  bool xtx_pending_ = false;
  static int nccl_unique_id(unsigned char* out128, std::string& e);
  int upload_xtx();
  // log-density pieces of the slot `rel` summed into `dev_red8` (+ all-reduce of the rank's own part); out3_host != NULL
  // also brings {loglik_w, logdetCi, failed factorisations} to the host (one synchronisation)
  int reduce_loglik(int rel, int* fail, double* dev_red8, double* out3_host);
  // ---- parameters (host copies of the small ones)
  dvec theta[2];
  double loglik_w[2] = {0, 0}, logdetCi[2] = {0, 0};
  int cur = 0;  // param_data = slot `cur`
  dvec Bcoeff;  // p x q
  dvec tausq_inv;
  HostRng rng;
  bool gram_stale = true;         // message Grams depend on the param slot's theta only
  bool pred_H_valid = false;
  bool alter_scratch = false;     // the alter slot holds a predict_new BUILD, not theta[alter]'s: rebuilt before it is read
  uint64_t sweep_counter = 0;
  // ---- device
  DevTree dt{};
  DevSlot ds[2]{};
  DevSlots dslots{};                // both slots + the chain state: what the kernels take
  ChainDev *d_mc = nullptr, *h_mc = nullptr;  // the chain state (st_chain.hpp) on the device and its pinned host mirror
  long long* d_rowkey = nullptr;    // node-major row -> row id in the whole problem (key of the device random streams)
  double* d_red_scratch = nullptr;  // partial sums and counters of loglik_reduce_kernel
  double* d_vrow = nullptr;         // per row of a reference block: -(L^-1 w)_r, written by an LLW pass (see launch_llw)
  double *d_xtx = nullptr, *d_bscratch = nullptr;   // XtX per outcome; scratch of the device beta step
  double *d_theta_mcmc = nullptr, *d_beta_mcmc = nullptr, *d_tausq_mcmc = nullptr, *d_yhat = nullptr;  // sample arrays of a device-resident run
  void* graph_exec_[2] = {nullptr, nullptr};  // cudaGraphExec_t of one device-resident iteration without / with prediction
  long long graph_key_[2] = {-1, -1};
  double* d_samp_ = nullptr;        // theta / beta / tausq samples of a device-resident run (kept between runs: the graphs hold its address)
  size_t samp_cap_ = 0;
  double graph_launches_[2] = {0, 0};
  double *d_w = nullptr, *d_xb = nullptr, *d_z = nullptr, *d_V = nullptr, *d_U = nullptr, *d_S = nullptr;
  double *d_Hpred = nullptr, *d_sdpred = nullptr;
  double *d_probe_sig = nullptr, *d_probe_smu = nullptr;  // Sigi_tot / Smu_tot probes (rioff / row0 indexed)
  double *d_scalars = nullptr, *h_scalars = nullptr;      // small result vector (pinned host mirror)
  double *d_partial = nullptr;
  double *d_bcoeff = nullptr, *d_tausq_inv = nullptr;
  int* d_fail = nullptr;
  int *d_grp_slot0 = nullptr, *d_grp_nn = nullptr;
  double* h_stage = nullptr;  // pinned n_all staging buffer
  cudaStream_t stream = nullptr, copy_stream = nullptr;
  cudaStream_t stream2 = nullptr;   // the early levels of a proposal's BUILD run here, underneath the Gibbs sweep
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_sweep = nullptr, ev_llw = nullptr, ev_acc = nullptr, ev_cond = nullptr,
              ev_early_llw = nullptr, ev_prop = nullptr, ev_zfree = nullptr;
  cudaStream_t stream3 = nullptr;   // the next iteration's proposal, drawn right after the accept step underneath the tail
  // LLW of the current slot on the second stream, underneath BUILD.  Off by default: measured on one B200 it gives 0.8 % at C4
  // and 2.3 % at C3 (the sweep of the HBM mostly displaces BUILD's own time) and makes LLW's event time meaningless;
  // ST_LLW_OVERLAP=1 enables it
  bool llw_overlap = false;
  bool overlap = true;              // ST_OVERLAP=0 disables
  int n_early_levels_ = 0;          // leading tree levels whose BUILD runs underneath the sweep (ST_EARLY_LEVELS overrides)
  long long* d_iperm = nullptr;     // boundary row -> node-major row
  cudaEvent_t ev[14]{};
  std::vector<void*> owned;  // device allocations to free
  // counters
  double n_launches = 0, f_alg = 0, f_exec = 0, n_cov = 0, f_alg_build = 0, f_exec_build = 0, b_alg_build = 0;
  std::string err;

  // ---- life cycle
  int init(std::string& e);  // bookkeeping + upload; returns st_status
  // ---- reference-named operations (spamtree_model.cpp)
  int theta_update(int slot, const double* th);
  int get_loglik_comps_w(int slot, double* out3);      // BUILD  :834-998
  int deal_with_w(const double* z, uint64_t seed);     // GIBBS  :1011-1226
  int get_loglik_w(int slot, double* out2);            // LLW    :781-826
  void accept_make_change();                           // :1432-1435
  int predict(bool theta_changed);                     // :1234-1358
  int gibbs_sample_beta(const double* zb, bool faithful_index);  // :1364-1391
  int gibbs_sample_tausq(const double* fixed);         // :1393-1417
  int get_w(double* out);
  int get_loglik_int(double* out);  // st_get_loglik_int
  int copy_store(int which, double* out, int64_t* n_rows, int32_t* n_samples);  // st_copy_store
  // a saved iteration's w (k = 0, un-permuted) or yhat (k = 1, device-resident chain only), in boundary order: written on
  // `stream` into `dev` (a slot of the device store) or, when dev is NULL, into co's staging slot k, then copied to `host`
  // (NULL: none) on the copy stream
  int save_rows(CopyOut& co, int k, double* dev, double* host);
  int set_w(const double* in);
  int get_xb(double* out);
  int set_tausq_inv(const double* t);
  int get_node_state(int slot, int u, const std::string& which, double* out, int64_t cap, int64_t* count);
  int get_index(const std::string& which, int u, int c, int64_t* out, int64_t cap, int64_t* count);
  int bench_iteration(const double* theta_prop, int do_swap, uint64_t seed, double* out3, float* ms_out);
  int sync();
  int set_widx_mode(bool faithful_index);
  // ---- the device-resident chain (rng_mode 1): spamtree_fit.cpp:167-391 without a host round trip per iteration
  int chain_run(const st_mcmc_opts& o, st_mcmc_out& out);
  // ---- prediction at new rows from saved samples (include/spamtree_b200.h: st_predict_new); from_store: the samples are
  // the last stored run's (st_predict_new_stored: ps carries only the seed), keep_draws: the draws go to the device store too
  int predict_new(const st_new_rows& rows, const st_pred_samples& ps, st_pred_out& out, bool from_store = false,
                  bool keep_draws = false);
  // ---- device sample store (st_keep_samples_on_device, st_summarize; DESIGN.md §5c)
  int keep_samples_on_device(int what);
  int summarize(int which, const double* probs, int n_probs, st_summary_out& out);
  int keep_mask = 0;                   // ST_KEEP_W | ST_KEEP_YHAT | ST_KEEP_LOGLIK_INT for the following device-resident runs
  DrawStore store;

 private:
  int phys(int slot) const { return slot ? 1 - cur : cur; }
  int build_bookkeeping(std::string& e);
  int build_layout(std::string& e);
  void bucket_groups(const std::vector<GroupSpec>& gs, const std::function<size_t(const GroupSpec&, int, int)>& need,
                     std::vector<int>& slot0, std::vector<int>& nn, std::vector<LevelInfo::BuildLaunch>& out) const;
  int upload(std::string& e);
  int launch_build_levels(int rel, int l0, int l1, bool no_density, cudaStream_t st);
  int complete_slot(int pslot);  // the deferred half of BUILD for the slot's childless levels, if pending
  int launch_deferred_half(int rel, const int* run_flag, cudaStream_t st);
  int push_slot_theta(int ps);   // host-driven path: theta[ps] and its covariance table into the device chain state
  int enqueue_gibbs(uint64_t seed, bool device_chain, bool draw = true, bool iloo = false);
  int enqueue_stats();
  int enqueue_iteration(const st_mcmc_opts& o, bool predicting, int accept_mode, bool draws_here, bool draws_next, int record_keep = 0);
  int push_chain_state(const st_mcmc_opts* o, uint64_t seed);
  int pull_chain_state();
  cudaEvent_t* timing_events_ = nullptr;
  bool deferred_[2] = {false, false};
  int refresh_grams(const int* run_flag = nullptr, cudaStream_t st = nullptr);
  int gibbs_launch_only(int* fail_ptr, bool iloo = false);
  // the integrated log-likelihood of the sweeps that form it (ST_KEEP_LOGLIK_INT; DESIGN.md §5f): node-major, n_all doubles,
  // NaN until a sweep writes them (the rows that are not observed stay NaN), then n_all doubles of y node-major with NaN at
  // the rows that are not observed, which tell the ILOO Gibbs kernel which rows to form.  Allocated and filled once.
  double* d_ll_int_ = nullptr;
  bool ll_int_valid_ = false;  // a sweep has formed it
  int alloc_loglik_int();
  int rowstats(bool faithful_index);
  std::vector<int> isref_host_;
  long long sd_total_ = 0;
  int llw_maxlen_ = 2;  // longest [w_pa ; w_u] any block stages in the LLW kernel
  int rowstat_blocks_ = 1;
  int draw_normals(uint64_t seed);
  int upload_rows(const double* boundary_order, double* dev);
  int cuda_fail(cudaError_t e, const char* what);
  std::vector<int> beta_widx_faithful, beta_widx_plain;
  int beta_widx_mode = -1;
  int stats_valid_mode_ = -1;  // row-index mode for which h_scalars holds the current beta / tausq statistics (-1: stale)
  int* d_obs_widx = nullptr;
};

// ---- several chains (st_summarize_chains, st_summarize_draws; DESIGN.md §5d).  chains_check: K, S and probs as both
// entry points refuse them (1), or K chains of S draws beyond one CTA's shared memory (4).  summarize_chains: src = K device
// pointers (a host array), chain c's draw (s, i) at src[c][s * n + i]; runs on st and synchronises it; outputs as
// st_chains_summary_out (NULL skipped, all NULL: the sizes only).  probs_check: n_probs >= 0 probabilities in [0, 1] (1)
int probs_check(const char* what, const double* probs, int n_probs, std::string& err);
int chains_check(const char* what, int K, int S, const double* probs, int n_probs, std::string& err);
int summarize_chains(const double* const* src, int64_t n, int K, int S, const double* probs, int n_probs, st_chains_summary_out& out,
                     cudaStream_t st, std::string& err);

// ---- model criteria (st_fit_criteria, st_fit_criteria_loglik; DESIGN.md §5e).  criteria_check: K, S and r_eff as both entry
// points refuse them (1), or K S draws beyond one CTA's shared memory (4).  fit_criteria: src = K device pointers (a host
// array), chain c's draw (s, i) at src[c][s * n + i]: w when `in` is given, else the log-likelihood itself; obs: n flags of
// the observed rows.  Runs on st and synchronises it; outputs and totals as st_fit_criteria_out (all NULL: the sizes only).
struct CritInputs {          // host arrays, rows in boundary order
  const double* y;           // n, NaN = missing
  const double* X;           // n x p, column-major
  const int64_t* mv_id;      // n, 1-based
  const double* beta;        // pooled draw g's p x q coefficients at beta[g p q ..), column-major
  const double* tausq;       // pooled draw g's q variances at tausq[g q ..)
  int p, q;
};
int criteria_check(const char* what, int K, int S, double r_eff, std::string& err);
int fit_criteria(const double* const* src, int64_t n, int K, int S, double r_eff, const std::vector<char>& obs, const CritInputs* in,
                 st_fit_criteria_out& out, cudaStream_t st, std::string& err);

}  // namespace st
