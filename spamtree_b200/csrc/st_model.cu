// st_model.cu — host side of the SpamTreeMV mirror: bookkeeping (spamtree_model.cpp:8-503 re-designed around ancestor
// chains), node-major layout, device state, and the reference-named operations that launch the kernels.
#include "st_model.hpp"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <numeric>

#include "../../include/spamtree_b200.h"
#include "st_kernels.cuh"

#include <chrono>
#include <dlfcn.h>
#include <nvtx3/nvToolsExt.h>  // header-only; the ranges cost nothing unless a profiler is attached (ncu --nvtx, nsys)

namespace st {

// ---- NCCL, resolved at run time: in a torch process dlopen returns the copy torch has already loaded
namespace {
struct NcclApi {
  typedef struct { char internal[128]; } UniqueId;
  int (*GetUniqueId)(UniqueId*) = nullptr;
  int (*CommInitRank)(void**, int, UniqueId, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
  std::string why;
  NcclApi() {
    void* h = nullptr;
    for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
      h = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
      if (h) break;
    }
    if (!h) { why = "libnccl.so.2 not found"; return; }
    GetUniqueId = (decltype(GetUniqueId))dlsym(h, "ncclGetUniqueId");
    CommInitRank = (decltype(CommInitRank))dlsym(h, "ncclCommInitRank");
    AllReduce = (decltype(AllReduce))dlsym(h, "ncclAllReduce");
    CommDestroy = (decltype(CommDestroy))dlsym(h, "ncclCommDestroy");
    GetErrorString = (decltype(GetErrorString))dlsym(h, "ncclGetErrorString");
    ok = GetUniqueId && CommInitRank && AllReduce && CommDestroy;
    if (!ok) why = "libnccl lacks a required symbol";
  }
};
NcclApi& nccl() { static NcclApi a; return a; }
constexpr int kNcclDouble = 8, kNcclSum = 0;  // ncclFloat64, ncclSum (nccl.h)
}  // namespace



// NVTX range over a scope: the phases of an iteration show up by name in a profiler's timeline / can be selected with
// `ncu --nvtx --nvtx-include "BUILD/"`
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

#define ST_CUDA(call, what)                                   \
  do {                                                        \
    cudaError_t _e = (call);                                  \
    if (_e != cudaSuccess) return cuda_fail(_e, what);        \
  } while (0)

int Model::cuda_fail(cudaError_t e, const char* what) {
  err = std::string("CUDA error in ") + what + ": " + cudaGetErrorString(e);
  return 2;  // ST_ERR_CUDA
}

// covariance_functions.cpp:34-92 / :113-135 -> per outcome-pair coefficients (make_covtab_hd, st_chain.hpp)
bool make_covtab(const double* theta, int n_theta, int q, CovTab& tab, std::string& err) {
  const int rc = make_covtab_hd(theta, n_theta, q, tab);
  if (rc == 1) err = "q outside 1..8";
  if (rc == 2) err = "theta has the wrong length for q";
  return rc == 0;
}

Model::~Model() {
  if (device < 0) return;
  cudaSetDevice(device);
  if (nccl_comm) { cudaStreamSynchronize(stream); nccl().CommDestroy(nccl_comm); nccl_comm = nullptr; }
  for (void* p : owned) cudaFree(p);
  store.release();
  if (h_scalars) cudaFreeHost(h_scalars);
  if (h_mc) cudaFreeHost(h_mc);
  for (void* g : graph_exec_) if (g) cudaGraphExecDestroy((cudaGraphExec_t)g);
  if (h_stage) cudaFreeHost(h_stage);
  for (auto& e : ev) if (e) cudaEventDestroy(e);
  if (copy_stream) cudaStreamDestroy(copy_stream);
  if (stream2) cudaStreamDestroy(stream2);
  if (stream3) cudaStreamDestroy(stream3);
  if (ev_prop) cudaEventDestroy(ev_prop);
  if (ev_zfree) cudaEventDestroy(ev_zfree);
  if (d_samp_) cudaFree(d_samp_);
  if (ev_fork) cudaEventDestroy(ev_fork);
  if (ev_join) cudaEventDestroy(ev_join);
  if (ev_sweep) cudaEventDestroy(ev_sweep);
  if (ev_acc) cudaEventDestroy(ev_acc);
  if (ev_cond) cudaEventDestroy(ev_cond);
  if (ev_early_llw) cudaEventDestroy(ev_early_llw);
  if (ev_llw) cudaEventDestroy(ev_llw);
  if (stream) cudaStreamDestroy(stream);
}

// ------------------------------------------------------------------------------------------------------ bookkeeping
int Model::build_bookkeeping(std::string& e) {
  const int nb = n_blocks;
  if ((int64_t)indexing.size() != nb || (int64_t)parents.size() != nb || (int64_t)children.size() != nb) { e = "CSR sizes do not match n_blocks"; return 1; }
  // the ABI promises status codes, not out-of-bounds reads: block ids of the edge lists must be block ids
  for (const CSR* c : {&parents, &children})
    for (int64_t v : c->idx)
      if (v < 0 || v >= nb) { e = "a parents / children list holds a block id outside 0..n_blocks-1"; return 1; }
  if ((int64_t)block_names.size() != nb || (int64_t)block_groups.size() != nb) { e = "block_names / block_groups do not match n_blocks"; return 1; }
  // na_ix_all, counts (spamtree_model.cpp:80-96)
  nobs_by_q.assign(q, 0);
  for (int64_t i = 0; i < n_all; i++) {
    if (mv_id[i] < 1 || mv_id[i] > q) { e = "mv_id outside 1..q"; return 1; }
    if (std::isfinite(y[i])) { na_ix_all.push_back(i); nobs_by_q[mv_id[i] - 1]++; }
  }
  n_obs = (int64_t)na_ix_all.size();
  // na_study :303-313
  block_ct_obs.assign(nb, 0);
  for (int b = 0; b < nb; b++)
    for (int64_t t = indexing.ptr[b]; t < indexing.ptr[b + 1]; t++) {
      const int64_t r = indexing.idx[t];
      if (r < 0 || r >= n_all) { e = "indexing row out of range"; return 1; }
      if (std::isfinite(y[r])) block_ct_obs[b]++;
    }
  // XtX :151-155 (over observed rows of each outcome)
  XtX.assign(q, SmallMat(p));
  for (int64_t i : na_ix_all) {
    SmallMat& M = XtX[mv_id[i] - 1];
    for (int a = 0; a < p; a++)
      for (int b = 0; b < p; b++) M(a, b) += X[i + (size_t)a * n_all] * X[i + (size_t)b * n_all];
  }
  // make_gibbs_groups :194-301
  dvec labels(block_groups);
  std::sort(labels.begin(), labels.end());
  labels.erase(std::unique(labels.begin(), labels.end()), labels.end());
  n_gibbs_groups = (int)labels.size();
  auto group_of = [&](int u) { return (int)(std::lower_bound(labels.begin(), labels.end(), block_groups[u]) - labels.begin()); };
  for (int i = 0; i < nb; i++) {  // :201-226
    const int u = (int)block_names[i] - 1;
    if (u < 0 || u >= nb) { e = "block name out of range"; return 1; }
    if (indexing.len(u) == 0) continue;
    for (int64_t t = parents.ptr[u]; t < parents.ptr[u + 1]; t++)
      if (block_groups[parents.idx[t]] == block_groups[u]) { e = "a block shares its group with a parent"; return 1; }
    for (int64_t t = children.ptr[u]; t < children.ptr[u + 1]; t++)
      if (block_groups[children.idx[t]] == block_groups[u]) { e = "a block shares its group with a child"; return 1; }
  }
  std::vector<ivec> temp(n_gibbs_groups);
  for (int i = 0; i < nb; i++) {
    const int u = (int)block_names[i] - 1;
    if (block_ct_obs[u] > 0) temp[group_of(u)].push_back(u);
  }
  n_actual_groups = 0;
  for (auto& t : temp) if (!t.empty()) n_actual_groups++;
  u_by_block_groups.assign(n_actual_groups, ivec());
  for (int g = 0; g < n_actual_groups; g++) u_by_block_groups[g] = temp[g];  // :257-260 (SURVEY App. D #3)
  for (int g = 0; g < n_actual_groups; g++)
    if (u_by_block_groups[g].empty()) { e = "an empty level precedes a non-empty one (reference assumes empties are last)"; return 1; }
  block_is_reference.assign(nb, 1);
  std::vector<char> in_nonref(nb, 0);
  for (size_t r = 0; r < res_is_ref.size(); r++)
    if (res_is_ref[r] == 0 && r < u_by_block_groups.size())
      for (int64_t u : u_by_block_groups[r]) in_nonref[u] = 1;
  for (int i = 0; i < nb; i++) {
    const int u = (int)block_names[i] - 1;
    if (block_ct_obs[u] > 0) {
      blocks_not_empty.push_back(u);
      if (in_nonref[u]) block_is_reference[u] = 0;
    } else {
      blocks_predicting.push_back(u);
      block_is_reference[u] = 0;
    }
  }
  if ((int)res_is_ref.size() < n_actual_groups) { e = "res_is_ref shorter than the number of levels"; return 1; }
  return 0;
}

// ------------------------------------------------------------------------------------------------------ layout
static inline long long pad2(long long v) { return (v + 1) & ~1LL; }

// BUILD launches of a list of work groups (slot s, nn sibling blocks, NT 8-column tiles): buckets by width (up to 4, 8, 16
// tiles) so that narrow groups are not launched with the shared memory and CTA size of the widest one, and the ring depth of
// each bucket; need(g, ns, nwarps) = shared memory of group g.  The groups go to (slot0, nn) in launch order.
void Model::bucket_groups(const std::vector<GroupSpec>& gs, const std::function<size_t(const GroupSpec&, int, int)>& need,
                          std::vector<int>& slot0, std::vector<int>& nn, std::vector<LevelInfo::BuildLaunch>& out) const {
  const int wmax = kBuildMaxThreads / 32;
  const size_t half_sm = (size_t)113 * 1024;
  for (int b = 0; b < 3; b++) {
    const int lo = (b == 0) ? 0 : (b == 1 ? 4 : 8), hi = (b == 0) ? 4 : (b == 1 ? 8 : 16);
    LevelInfo::BuildLaunch bl;
    bl.grp0 = (int)slot0.size();
    size_t need1 = 0, need2 = 0;
    int maxNT = 1;
    for (const GroupSpec& g : gs)
      if (g.NT > lo && g.NT <= hi) maxNT = std::max(maxNT, g.NT);
    const int nw = std::min(wmax, std::max(4, (2 * maxNT) & ~3));
    for (const GroupSpec& g : gs)
      if (g.NT > lo && g.NT <= hi) {
        slot0.push_back(g.s); nn.push_back(g.nn);
        need1 = std::max(need1, need(g, 1, nw));
        need2 = std::max(need2, need(g, 2, nw));
      }
    bl.ngrp = (int)slot0.size() - bl.grp0;
    if (bl.ngrp == 0) continue;
    // ring depth: double-buffered when it fits; single-buffered when that lets two CTAs share an SM (they overlap instead)
    if (force_build_ns == 1 || force_build_ns == 2) bl.ns = (force_build_ns == 2 && need2 <= smem_budget) ? 2 : 1;
    else if (need2 <= std::min(half_sm, smem_budget)) bl.ns = 2;  // (a budget set below half an SM holds for the ring too)
    else if (need1 <= half_sm) bl.ns = 1;
    else bl.ns = (need2 <= smem_budget) ? 2 : 1;
    bl.smem = (bl.ns == 2) ? need2 : need1;
    bl.threads = 32 * nw;
    out.push_back(bl);
  }
}

int Model::build_layout(std::string& e) {
  const int nb = n_blocks;
  slot_of_block.assign(nb, -1);
  block_of_slot.clear();
  levels.clear();
  auto chain_ok = [&](int u, std::string& why) {
    // parents(u) must be parents(lp) followed by lp (tree_dep.cpp:113-119 gives exactly that), all reference blocks
    const int64_t np = parents.len(u);
    if (np == 0) return true;
    const int lp = (int)parents.back(u);
    if (slot_of_block[lp] < 0 || block_ct_obs[lp] == 0) { why = "a parent is not an observed block of a shallower level"; return false; }
    if (!block_is_reference[lp]) { why = "a parent is not a reference block"; return false; }
    if (limited) {  // limited trees: the direct parent only (make_edges_limited, tree_dep.cpp:133-186)
      if (np != 1) { why = "limited_tree = TRUE: a block lists more than one parent (use make_edges_limited)"; return false; }
      return true;
    }
    if (parents.len(lp) != np - 1 || !std::equal(parents.row(lp), parents.row(lp) + (np - 1), parents.row(u))) {
      why = "parent set is not the ancestor chain of its last parent";
      return false;
    }
    return true;
  };
  auto order_level = [&](ivec us) {
    std::sort(us.begin(), us.end(), [&](int64_t a, int64_t b) {
      const int pa = parents.len(a) ? slot_of_block[parents.back(a)] : -1;
      const int pb = parents.len(b) ? slot_of_block[parents.back(b)] : -1;
      if (pa != pb) return pa < pb;
      return a < b;
    });
    return us;
  };
  std::string why;
  for (int g = 0; g < n_actual_groups; g++) {
    for (int64_t u : u_by_block_groups[g])
      if (!chain_ok((int)u, why)) { e = "unsupported DAG: " + why; return 4; }
    ivec us = order_level(u_by_block_groups[g]);
    LevelInfo L;
    L.slot0 = (int)block_of_slot.size();
    L.nslots = (int)us.size();
    L.is_ref = res_is_ref[g] == 1 ? 1 : 0;  // indexed by group like spamtree_model.cpp:890,1037
    for (int64_t u : us) { slot_of_block[u] = (int)block_of_slot.size(); block_of_slot.push_back((int)u); }
    levels.push_back(L);
  }
  n_obs_nodes = (int)block_of_slot.size();
  {
    for (int64_t u : blocks_predicting) {
      if (parents.len(u) == 0) { e = "a block without observations has no parents"; return 1; }
      if (!chain_ok((int)u, why)) { e = "unsupported DAG (prediction block): " + why; return 4; }
    }
    ivec us = order_level(blocks_predicting);
    pred_level = LevelInfo();
    pred_level.slot0 = n_obs_nodes;
    pred_level.nslots = (int)us.size();
    pred_level.is_ref = 0;
    for (int64_t u : us) { slot_of_block[u] = (int)block_of_slot.size(); block_of_slot.push_back((int)u); }
  }
  n_nodes = (int)block_of_slot.size();
  // every observed block must list its parents' children consistently (used by this_is_jth_child, :411-417)
  for (int s = 0; s < n_obs_nodes; s++) {
    const int u = block_of_slot[s];
    for (int64_t t = parents.ptr[u]; t < parents.ptr[u + 1]; t++) {
      const int64_t pa = parents.idx[t];
      const int64_t* b = children.row(pa);
      const int64_t* en = b + children.len(pa);
      // make_edges returns sorted lists (arma::intersect, tree_dep.cpp:106); fall back to a scan for unsorted input
      if (!std::binary_search(b, en, (int64_t)u) && std::find(b, en, (int64_t)u) == en) {
        e = "children lists are inconsistent with parents lists";
        return 1;
      }
    }
    if (!block_is_reference[u] && children.len(u) > 0) { e = "a non-reference block has children"; return 4; }
  }
  // rows: node-major permutation
  perm.clear();
  perm.reserve(n_all);
  h_m.assign(n_nodes, 0); h_row0.assign(n_nodes, 0); h_k.assign(n_nodes, 0); h_P.assign(n_nodes, 0);
  h_chain_off.assign(n_nodes, 0); h_lastpar.assign(n_nodes, -1);
  for (int s = 0; s < n_nodes; s++) {
    const int u = block_of_slot[s];
    h_row0[s] = (int)perm.size();
    h_m[s] = (int)indexing.len(u);
    for (int64_t t = indexing.ptr[u]; t < indexing.ptr[u + 1]; t++) perm.push_back(indexing.idx[t]);
  }
  if ((int64_t)perm.size() != n_all) { e = "indexing does not cover every row exactly once"; return 1; }
  iperm.assign(n_all, -1);
  for (int64_t i = 0; i < n_all; i++) {
    if (iperm[perm[i]] != -1) { e = "a row belongs to two blocks"; return 1; }
    iperm[perm[i]] = i;
  }
  // chains and storage offsets
  h_chain.clear(); h_chain_poff.clear(); h_chain_uoff.clear();
  h_gs.assign(n_nodes, 0);
  h_moff.assign(n_nodes, -1);
  h_goff.assign(n_nodes, 0); h_rioff.assign(n_nodes, 0); h_voff.assign(n_nodes, 0); h_uoff.assign(n_nodes, 0); h_soff.assign(n_nodes, -1);
  g_total = ri_total = v_total = u_total = s_total = gpred_total = 0;
  std::vector<long long> h_usize(n_nodes, 0);
  long long sd_total = 0;
  std::vector<int> isref(n_nodes, 0);
  auto poff_check = [&](int u) {
    long long t = 0;
    for (int64_t x = parents.ptr[u]; x < parents.ptr[u + 1]; x++) t += indexing.len(parents.idx[x]);
    return t;
  };
  for (int s = 0; s < n_nodes; s++) {
    const int u = block_of_slot[s];
    const bool pred = s >= n_obs_nodes;
    const int kk = (int)parents.len(u);
    if (kk > 32) { e = "ancestor chains longer than 32 are not supported"; return 4; }
    if (limited && kk > 1) { e = "limited_tree = TRUE: a block lists more than one parent (use make_edges_limited)"; return 1; }
    if (!pred && poff_check(u) > kLlwMaxP) { e = "a parent set larger than 1024 rows is not supported"; return 4; }
    h_k[s] = kk;
    h_chain_off[s] = (int)h_chain.size();
    int poff = 0;
    long long uo = 0;
    for (int j = 0; j < kk; j++) {
      const int a = slot_of_block[parents.idx[parents.ptr[u] + j]];
      h_chain.push_back(a);
      h_chain_poff.push_back(poff);
      h_chain_uoff.push_back((int)uo);
      poff += h_m[a];
      uo += pad2((long long)h_m[a] * h_m[a]);
    }
    h_P[s] = poff;
    // the block's rows of the chain's inverse Cholesky factor: [ G (P) | -Ri (m, reference blocks) | 0 ]
    h_gs[s] = g_stride(poff, h_m[s], (!pred && block_is_reference[u]) ? 1 : 0);
    const long long boff = (long long)h_m[s] * h_gs[s];
    if (kk) h_lastpar[s] = h_chain.back();
    if (!pred) {
      isref[s] = block_is_reference[u] ? 1 : 0;
      h_goff[s] = g_total; g_total += boff;
      if (limited && isref[s]) { h_moff[s] = g_total; g_total += (long long)h_m[s] * ((h_m[s] + 3) & ~3); }  // marginal factor rows
      h_rioff[s] = ri_total; ri_total += isref[s] ? (long long)h_m[s] * tile_rs(h_m[s]) : pad2(h_m[s]);
      h_voff[s] = v_total; v_total += pad2(poff);
      h_usize[s] = uo;
    } else {
      h_goff[s] = gpred_total; gpred_total += boff;
      h_rioff[s] = sd_total; sd_total += pad2(h_m[s]);
    }
  }
  // partition: the deepest replicated level pulls its children's messages through one pseudo child per block, filled
  // by an all-reduce over the ranks (its real children live on several ranks)
  n_slots_total = n_nodes;
  n_top_slots = 0;
  std::vector<char> is_front(n_nodes, 0);
  h_front_pseudo.clear(); h_front_c0.clear(); h_front_c1.clear(); h_front_vlen.clear(); h_front_ulen.clear();
  v_front0 = v_total;
  if (part) {
    if (n_top_levels < 0 || n_top_levels >= (int)levels.size()) { e = "partition: n_top_levels out of range"; return 1; }
    for (int g = 0; g < n_top_levels; g++) n_top_slots += levels[g].nslots;
    n_top_rows = (n_top_slots < n_nodes) ? h_row0[n_top_slots] : (int)n_all;
    if (n_top_levels >= 1) {
      const LevelInfo& FL = levels[n_top_levels - 1];
      const LevelInfo& CL = levels[n_top_levels];
      if (!FL.is_ref) { e = "partition: the deepest replicated level must be a reference level"; return 1; }
      int c = CL.slot0;
      for (int dd = FL.slot0; dd < FL.slot0 + FL.nslots; dd++) {
        is_front[dd] = 1;
        const int ps = n_slots_total++;
        const int c0 = c;
        while (c < CL.slot0 + CL.nslots && h_lastpar[c] == dd) c++;
        // the pseudo child looks like a child of dd with no rows: chain = chain(dd) + dd
        h_m.push_back(0); h_row0.push_back(0); isref.push_back(0); h_lastpar.push_back(dd);
        // (limited trees: a child lists its direct parent only, tree_dep.cpp:133-186 — so does the pseudo child)
        const int kps = limited ? 0 : h_k[dd];
        h_k.push_back(kps + 1);
        h_chain_off.push_back((int)h_chain.size());
        int poff = 0;
        long long uo = 0;
        for (int j = 0; j <= kps; j++) {
          const int a = (j < kps) ? h_chain[h_chain_off[dd] + j] : dd;
          h_chain.push_back(a); h_chain_poff.push_back(poff); h_chain_uoff.push_back((int)uo);
          poff += h_m[a];
          uo += pad2((long long)h_m[a] * h_m[a]);
        }
        h_P.push_back(poff);
        h_goff.push_back(0); h_rioff.push_back(0); h_soff.push_back(-1); h_gs.push_back(0); h_moff.push_back(-1);
        h_voff.push_back(v_total); v_total += pad2(poff);
        h_uoff.push_back(0); h_usize.push_back(uo);
        h_front_pseudo.push_back(ps); h_front_c0.push_back(c0); h_front_c1.push_back(c);
        h_front_vlen.push_back(poff); h_front_ulen.push_back((int)uo);
      }
      if (c != CL.slot0 + CL.nslots) { e = "partition: a block of the cut level has no replicated parent"; return 1; }
    }
    v_front_len = v_total - v_front0;
  }
  // direct children among observed nodes (contiguous by construction of the slot order)
  h_child_ptr.assign(n_slots_total + 1, 0);
  for (int s = 0; s < n_obs_nodes; s++)
    if (h_lastpar[s] >= 0 && !is_front[h_lastpar[s]]) h_child_ptr[h_lastpar[s] + 1]++;
  for (size_t i = 0; i < h_front_pseudo.size(); i++) h_child_ptr[h_lastpar[h_front_pseudo[i]] + 1]++;
  for (int s = 0; s < n_slots_total; s++) h_child_ptr[s + 1] += h_child_ptr[s];
  h_child_idx.assign(h_child_ptr[n_slots_total], 0);
  {
    std::vector<int> fill(h_child_ptr.begin(), h_child_ptr.end() - 1);
    for (int s = 0; s < n_obs_nodes; s++)
      if (h_lastpar[s] >= 0 && !is_front[h_lastpar[s]]) h_child_idx[fill[h_lastpar[s]]++] = s;
    for (size_t i = 0; i < h_front_pseudo.size(); i++) h_child_idx[fill[h_lastpar[h_front_pseudo[i]]]++] = h_front_pseudo[i];
  }
  for (int s = 0; s < n_obs_nodes; s++)
    if (h_child_ptr[s + 1] > h_child_ptr[s]) { h_soff[s] = s_total; s_total += pad2((long long)h_m[s] * h_m[s]); }
  // message Grams: a childless block that is pulled by an ordinary parent is "fused" — the parent forms its tiles from
  // the block's rows on the fly (gram_level_kernel) and they are never stored.  Blocks under a replicated frontier block
  // keep theirs (frontier_sum_kernel adds them up for the all-reduce).
  h_ufused.assign(n_slots_total, 0);
  for (int s = 0; s < n_obs_nodes; s++)
    h_ufused[s] = (h_child_ptr[s + 1] == h_child_ptr[s] && h_lastpar[s] >= 0 && !is_front[h_lastpar[s]]) ? 1 : 0;
  u_total = 0;
  for (int s = 0; s < n_obs_nodes; s++)
    if (!h_ufused[s]) { h_uoff[s] = u_total; u_total += h_usize[s]; }
  u_front0 = u_total;
  for (int s = n_nodes; s < n_slots_total; s++) { h_uoff[s] = u_total; u_total += h_usize[s]; }
  u_front_len = u_total - u_front0;
  isref_host_ = isref;
  llw_maxlen_ = 2;
  for (int s = 0; s < n_obs_nodes; s++) llw_maxlen_ = std::max(llw_maxlen_, h_P[s] + h_m[s]);
  sd_total_ = sd_total;

  // BUILD work groups: runs of sibling blocks (they share their ancestor chain), at most max_group_cols columns
  // (one warp per 8 columns) and sized to the shared-memory budget
  h_grp_slot0.clear(); h_grp_nn.clear();
  auto group_plan = [&](int s, int nn, int mode, int ns, int nwarps, int xcol) {
    int ncols = xcol, sumRb = 0, maxmd = 1;
    for (int d = 0; d < nn; d++) {
      ncols += h_m[s + d];
      if (mode == 0) sumRb += (limited ? 2 : 1) * rb_doubles(h_m[s + d]);  // limited trees factorise K_uu as well
      maxmd = std::max(maxmd, h_m[s + d]);
    }
    return build_plan(h_P[s], ncols, sumRb, maxmd, ns, mode == 0 ? std::min((limited ? 2 : 1) * nn, kBuildMaxThreads / 32) : 0, nwarps);
  };
  auto make_groups = [&](LevelInfo& L, int mode) -> int {
    L.grp0 = (int)h_grp_slot0.size();
    L.smem_gibbs = 0;
    L.build_launches.clear();
    const int end = L.slot0 + L.nslots;
    const int col_cap = std::min(max_group_cols, kMaxGroupCols);
    // A level with fewer blocks than the GPU has SMs is a latency chain, not a throughput problem: smaller groups (down to
    // one block per CTA) shorten every phase of the chain and cost nothing, the other SMs are idle anyway.
    const int nn_cap = (spread_ctas > 0) ? std::max(1, std::min(kMaxGroupNodes, (L.nslots + spread_ctas - 1) / spread_ctas)) : kMaxGroupNodes;
    L.deferrable = false;
    if (mode == 1 && !keep_H && defer_leaves) {
      L.deferrable = L.nslots > 0;
      for (int t = L.slot0; t < end; t++)
        if (h_child_ptr[t + 1] > h_child_ptr[t] || h_lastpar[t] < 0) L.deferrable = false;
    }
    const int wmax = kBuildMaxThreads / 32;
    // the deferred scheme carries w_pa as one extra panel column: a block that fits one work group only without it (a leaf
    // of 128 rows, or one at the edge of the shared-memory budget) keeps the whole level on the eager scheme
    if (L.deferrable)
      for (int t = L.slot0; t < end && L.deferrable; t++) {
        const BuildPlan pl = group_plan(t, 1, mode, 1, wmax, 1);
        if (pl.total > smem_budget || pl.NCp > kMaxGroupCols) L.deferrable = false;
      }
    const int xcol = L.deferrable ? 1 : 0;
    std::vector<GroupSpec> gs;
    int s = L.slot0;
    while (s < end) {
      int nn = 0;
      BuildPlan best{};
      while (s + nn < end && nn < nn_cap) {
        const int t = s + nn;
        if (nn > 0 && (h_lastpar[s] < 0 || h_lastpar[t] != h_lastpar[s])) break;  // roots never share a chain
        const BuildPlan pl = group_plan(s, nn + 1, mode, 1, wmax, xcol);
        if (pl.total > smem_budget || pl.NCp > kMaxGroupCols || (nn > 0 && pl.NCp > col_cap)) break;
        best = pl;
        nn++;
      }
      if (nn == 0) {
        e = "a block is too large for one BUILD work group (m=" + std::to_string(h_m[s]) + ", P=" + std::to_string(h_P[s]) + ")";
        return 4;
      }
      gs.push_back({s, nn, best.NT});
      L.maxNC = std::max(L.maxNC, best.NCp);
      s += nn;
    }
    bucket_groups(gs, [&](const GroupSpec& g, int ns, int nw) { return group_plan(g.s, g.nn, mode, ns, nw, xcol).total; }, h_grp_slot0,
                  h_grp_nn, L.build_launches);
    L.ngrp = (int)h_grp_slot0.size() - L.grp0;
    for (int t = L.slot0; t < end; t++) {
      L.maxP = std::max(L.maxP, h_P[t]); L.maxm = std::max(L.maxm, h_m[t]); L.maxk = std::max(L.maxk, h_k[t]);
      L.smem_gibbs = std::max(L.smem_gibbs, gibbs_smem_bytes(L.is_ref, h_m[t], h_P[t], h_k[t]));
    }
    if (mode != 2 && L.smem_gibbs > 227 * 1024) { e = "a block is too large for the Gibbs kernel's shared memory"; return 4; }
    if (mode != 2) {  // gram_level_kernel: rows staged per chunk (own rows + the rows of the fused children)
      int ldx = 2, maxrows = 1, maxitems = 1;
      long long tiles = 2;
      L.gram_skip = true;
      for (int t = L.slot0; t < end; t++) {
        if (h_ufused[t]) continue;
        L.gram_skip = false;
        int rows = h_m[t];
        for (int c = h_child_ptr[t]; c < h_child_ptr[t + 1]; c++) if (h_ufused[h_child_idx[c]]) rows += h_m[h_child_idx[c]];
        maxrows = std::max(maxrows, rows);
        ldx = std::max(ldx, (h_P[t] + h_m[t] + 1) & ~1);
        long long td = (long long)h_m[t] * h_m[t];
        int items = ((h_m[t] + 4) / 5) * ((h_m[t] + 4) / 5 + 1) / 2;
        for (int j = 0; j < h_k[t]; j++) {
          const long long mj = h_m[h_chain[h_chain_off[t] + j]];
          td += mj * mj;
          items += (int)(((mj + 4) / 5) * ((mj + 4) / 5 + 1) / 2);
        }
        tiles = std::max(tiles, (td + 1) & ~1LL);
        maxitems = std::max(maxitems, items);
      }
      L.gram_maxrows = maxrows;
      L.gram_maxitems = maxitems;
      if (tiles * 8 > 160 * 1024) { e = "a block's message Gram tiles do not fit the Gram kernel's shared memory"; return 4; }
      L.gram_ldx = ldx;
      L.gram_tiles = (int)tiles;
      // the assembled tiles take the place of the staged rows when every (tile, sub-block) item has its own thread: the
      // accumulators live in registers until the last row has been consumed
      // One thread per item, in whole warps.  The kernel needs ~128 registers per thread, so a 128-thread CTA can have
      // four co-resident CTAs per SM where a 256-thread CTA has two: the staged chunk is sized for that many (the kernel is
      // latency-bound: load, compute and store phases of different CTAs overlap).
      L.gram_threads = std::min(kGramThreads, std::max(64, (maxitems + 31) & ~31));
      if (L.nslots <= 2 * n_sm) L.gram_threads = kGramThreads;  // a level that does not fill the GPU is a latency chain: widest CTA
      L.gram_stage_off = (maxitems <= L.gram_threads) ? 0 : (int)tiles;
      const size_t fixed = (size_t)L.gram_stage_off * 8;
      const int ctas = std::max(1, std::min(8, 65536 / (128 * L.gram_threads)));
      size_t room = (size_t)(228 - ctas) * 1024 / ctas - 9 * 1024;  // per CTA: its share of the SM minus the static part
      if (const char* v = getenv("ST_GRAM_ROOM")) room = (size_t)atol(v);
      room = std::max(room, std::max((size_t)tiles * 8, fixed + (size_t)ldx * 8));
      room -= fixed;
      L.gram_rch = (int)std::max<size_t>(1, std::min<size_t>(std::min(maxrows, kGramMaxRows), room / ((size_t)ldx * 8)));
    }
    return 0;
  };
  for (auto& L : levels) { int rc = make_groups(L, L.is_ref ? 0 : 1); if (rc) return rc; }
  // the leading levels whose BUILD is a chain of small launches (fewer work groups than SMs): built underneath the Gibbs
  // sweep by the device-resident iteration; never the deepest level.  Measured on C4 / one B200 (ms per iteration): no
  // overlap 7.18, levels 0-4 (<= 128 groups) 7.17, + level 5 (256 groups) 7.21, + level 6 7.34, everything but the leaves 7.42
  // — a level that fills the GPU only competes with the sweep; C1 (n = 625): 4 998 -> 6 455 it/s end to end
  // A rank of a partitioned run holds a fraction of the big levels and is latency-dominated: there the threshold is four
  // waves of work groups (C4 on 8 B200: 577 it/s without overlap, 607 with the one-wave threshold, 639 with levels up to
  // 512 groups early; on one GPU the wider threshold costs 0.5 %).
  const int early_thr = (part ? 4 : 1) * n_sm;
  n_early_levels_ = 0;
  while (n_early_levels_ + 1 < (int)levels.size() && levels[n_early_levels_].ngrp <= early_thr && !levels[n_early_levels_].deferrable)
    n_early_levels_++;
  // On one GPU a big tree gains nothing from the overlap (C4: 7.17 vs 7.18 ms, C3: +1 %) — the sweep and the BUILD both fill
  // the machine — and its per-phase event times stay attributable without it: the overlap is for the latency-dominated
  // cases, small trees (C1: +30 %, C2: +35 % end to end) and the ranks of a partition (C4 on 8 B200: +11 %)
  if (!part && n_obs_nodes > 16384) n_early_levels_ = 0;
  // (ST_EARLY_LEVELS = the number of levels: the whole BUILD underneath the sweep, the childless level's log-density pieces
  // from its parked Z; not for limited trees, whose children do not stream the rows LLW reads)
  if (const char* v = getenv("ST_EARLY_LEVELS")) n_early_levels_ = std::max(0, std::min(atoi(v), (int)levels.size() - (limited ? 1 : 0)));
  { int rc = make_groups(pred_level, 2); if (rc) return rc; }

  // work counters per iteration (SURVEY §8d formulas on the actual tree)
  f_alg = f_exec = n_cov = f_alg_build = f_exec_build = b_alg_build = 0;
  for (int s = 0; s < n_obs_nodes; s++) {
    const double m = h_m[s], P = h_P[s], rho = isref[s], chi = (h_child_ptr[s + 1] > h_child_ptr[s]) ? 1.0 : 0.0;
    const double C = (double)children.len(block_of_slot[s]);
    const double fb = 2 * m * P * P + rho * (2 * m * m * P + m * m * m + 2 * m * P + 2 * m * m) + rho * chi * (m * m * P + std::pow(P + m, 3) / 3) + (1 - rho) * (4 * m * P);
    const double fg = rho * (2 * P * m * m + C * m * m + 2 * m * m * m / 3 + 2 * m * P + C * m + 4 * m * m + 2 * P * P * m + 2 * P * P + 2 * P * m) +
                      (1 - rho) * (3 * m * P + 2 * P * P * m + 2 * P * P + 2 * P * m + 10 * m);
    const double fl = 2 * m * P + rho * 2 * m * m + (1 - rho) * 2 * m;
    f_alg += fb + fg + fl;
    f_alg_build += fb;
    f_exec_build += 2 * m * P * P + rho * (2 * m * m * P + m * m * P + 2 * m * m * m / 3) + (1 - rho) * 3 * m * P + 2 * m * P;
    b_alg_build += 8 * (m * P + rho * m * m + (1 - rho) * m);  // compulsory output of BUILD: G and Ri of the slot
    // lean formulation actually executed: Z (mP^2) + H' (mP^2) + Z'Z (rho m^2 P, else mP) + G (rho m^2 P/ else mP) + chol/inv + Gibbs/LLW matvecs
    f_exec += 2 * m * P * P + rho * (2 * m * m * P + m * m * P + 2 * m * m * m / 3) + (1 - rho) * 3 * m * P + 2 * m * P +
              (4 * m * P + rho * (2 * m * m * m / 3 + 4 * m * m)) + (2 * m * P + rho * m * m);
    n_cov += P * m + rho * m * (m + 1) / 2 + (1 - rho) * m;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------------ upload
template <class T>
static cudaError_t dev_upload(const std::vector<T>& h, T*& d, std::vector<void*>& owned) {
  d = nullptr;
  const size_t bytes = std::max<size_t>(h.size(), 1) * sizeof(T);
  cudaError_t e = cudaMalloc((void**)&d, bytes);
  if (e != cudaSuccess) return e;
  owned.push_back(d);
  if (!h.empty()) e = cudaMemcpy(d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
  return e;
}
static cudaError_t dev_zeros(double*& d, long long n, std::vector<void*>& owned) {
  d = nullptr;
  const size_t bytes = (size_t)std::max<long long>(n, 1) * sizeof(double);
  cudaError_t e = cudaMalloc((void**)&d, bytes);
  if (e != cudaSuccess) return e;
  owned.push_back(d);
  return cudaMemset(d, 0, bytes);
}

int Model::upload(std::string& e) {
  (void)e;
  ST_CUDA(cudaSetDevice(device), "cudaSetDevice");
  {
    // the main stream outranks the second one: when both have thread blocks pending, those of the Gibbs sweep (a chain of
    // short launches) are dispatched before those of the BUILD levels that run underneath it
    int lo = 0, hi = 0;
    ST_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi), "cudaDeviceGetStreamPriorityRange");
    ST_CUDA(cudaStreamCreateWithPriority(&stream, cudaStreamNonBlocking, hi), "cudaStreamCreate");
    ST_CUDA(cudaStreamCreateWithPriority(&stream2, cudaStreamNonBlocking, lo), "cudaStreamCreate");
    ST_CUDA(cudaStreamCreateWithPriority(&stream3, cudaStreamNonBlocking, lo), "cudaStreamCreate");
    ST_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking), "cudaStreamCreate");  // saved rows (CopyOut)
  }
  ST_CUDA(cudaEventCreateWithFlags(&ev_prop, cudaEventDisableTiming), "cudaEventCreate");
  ST_CUDA(cudaEventCreateWithFlags(&ev_zfree, cudaEventDisableTiming), "cudaEventCreate");
  ST_CUDA(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming), "cudaEventCreate");
  ST_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming), "cudaEventCreate");
  ST_CUDA(cudaEventCreateWithFlags(&ev_acc, cudaEventDisableTiming), "cudaEventCreate");
  ST_CUDA(cudaEventCreateWithFlags(&ev_cond, cudaEventDisableTiming), "cudaEventCreate");
  ST_CUDA(cudaEventCreateWithFlags(&ev_early_llw, cudaEventDisableTiming), "cudaEventCreate");
  ST_CUDA(cudaEventCreateWithFlags(&ev_sweep, cudaEventDisableTiming), "cudaEventCreate");
  ST_CUDA(cudaEventCreateWithFlags(&ev_llw, cudaEventDisableTiming), "cudaEventCreate");
  for (auto& x : ev) ST_CUDA(cudaEventCreate(&x), "cudaEventCreate");
  // per row
  dvec cx(n_all), cy(n_all), yy(n_all), Xp((size_t)n_all * p), xb(n_all, 0.0);
  std::vector<int> mvq(n_all);
  for (int64_t i = 0; i < n_all; i++) {
    const int64_t b = perm[i];
    cx[i] = coords[b]; cy[i] = coords[b + n_all];
    mvq[i] = (int)mv_id[b] - 1;
    yy[i] = std::isfinite(y[b]) ? y[b] : 0.0;  // spamtree_model.cpp:146
    for (int a = 0; a < p; a++) Xp[i + (size_t)a * n_all] = X[b + (size_t)a * n_all];
    double s = 0;  // XB = X * beta_in for every outcome (:124-129)
    for (int a = 0; a < p; a++) s += X[b + (size_t)a * n_all] * Bcoeff[a + (size_t)mvq[i] * p];
    xb[i] = s;
  }
  double *d_cx, *d_cy, *d_y, *d_X;
  int *d_mvq, *d_m, *d_row0, *d_isref, *d_k, *d_P, *d_choff, *d_cptr, *d_cidx, *d_chain, *d_cpoff, *d_cuoff, *d_gs;
  long long *d_goff, *d_rioff, *d_voff, *d_uoff, *d_soff;
  ST_CUDA(dev_upload(cx, d_cx, owned), "upload cx");
  ST_CUDA(dev_upload(cy, d_cy, owned), "upload cy");
  ST_CUDA(dev_upload(yy, d_y, owned), "upload y");
  ST_CUDA(dev_upload(Xp, d_X, owned), "upload X");
  ST_CUDA(dev_upload(mvq, d_mvq, owned), "upload mv");
  ST_CUDA(dev_upload(h_m, d_m, owned), "upload m");
  ST_CUDA(dev_upload(h_row0, d_row0, owned), "upload row0");
  ST_CUDA(dev_upload(isref_host_, d_isref, owned), "upload isref");
  ST_CUDA(dev_upload(h_k, d_k, owned), "upload k");
  ST_CUDA(dev_upload(h_P, d_P, owned), "upload P");
  int* d_lastpar;
  ST_CUDA(dev_upload(h_lastpar, d_lastpar, owned), "upload lastpar");
  ST_CUDA(dev_upload(h_chain_off, d_choff, owned), "upload chain_off");
  ST_CUDA(dev_upload(h_goff, d_goff, owned), "upload goff");
  ST_CUDA(dev_upload(h_gs, d_gs, owned), "upload gs");
  long long* d_moff;
  ST_CUDA(dev_upload(h_moff, d_moff, owned), "upload moff");
  ST_CUDA(dev_upload(h_rioff, d_rioff, owned), "upload rioff");
  ST_CUDA(dev_upload(h_voff, d_voff, owned), "upload voff");
  ST_CUDA(dev_upload(h_uoff, d_uoff, owned), "upload uoff");
  ST_CUDA(dev_upload(h_soff, d_soff, owned), "upload soff");
  ST_CUDA(dev_upload(h_child_ptr, d_cptr, owned), "upload child_ptr");
  ST_CUDA(dev_upload(h_child_idx, d_cidx, owned), "upload child_idx");
  int* d_ufused;
  ST_CUDA(dev_upload(h_ufused, d_ufused, owned), "upload ufused");
  ST_CUDA(dev_upload(h_chain, d_chain, owned), "upload chain");
  ST_CUDA(dev_upload(h_chain_poff, d_cpoff, owned), "upload chain_poff");
  ST_CUDA(dev_upload(h_chain_uoff, d_cuoff, owned), "upload chain_uoff");
  ST_CUDA(dev_upload(h_grp_slot0, d_grp_slot0, owned), "upload groups");
  ST_CUDA(dev_upload(h_grp_nn, d_grp_nn, owned), "upload groups");
  ST_CUDA(dev_upload(h_front_pseudo, d_front_pseudo, owned), "upload frontier");
  ST_CUDA(dev_upload(h_front_c0, d_front_c0, owned), "upload frontier");
  ST_CUDA(dev_upload(h_front_c1, d_front_c1, owned), "upload frontier");
  ST_CUDA(dev_upload(h_front_vlen, d_front_vlen, owned), "upload frontier");
  ST_CUDA(dev_upload(h_front_ulen, d_front_ulen, owned), "upload frontier");
  dt.cx = d_cx; dt.cy = d_cy; dt.mvq = d_mvq; dt.y = d_y; dt.X = d_X;
  dt.m = d_m; dt.row0 = d_row0; dt.isref = d_isref; dt.k = d_k; dt.P = d_P; dt.lastpar = d_lastpar; dt.chain_off = d_choff;
  dt.goff = d_goff; dt.gs = d_gs; dt.moff = d_moff; dt.limited = limited ? 1 : 0; dt.rioff = d_rioff; dt.voff = d_voff; dt.uoff = d_uoff; dt.soff = d_soff;
  dt.child_ptr = d_cptr; dt.child_idx = d_cidx; dt.ufused = d_ufused;
  dt.chain = d_chain; dt.chain_poff = d_cpoff; dt.chain_uoff = d_cuoff;
  for (int s = 0; s < 2; s++) {
    ST_CUDA(dev_zeros(ds[s].G, g_total, owned), "alloc G");
    if (keep_H) ST_CUDA(dev_zeros(ds[s].H, g_total, owned), "alloc H"); else ds[s].H = nullptr;
    ST_CUDA(dev_zeros(ds[s].Ri, ri_total, owned), "alloc Ri");
    ST_CUDA(dev_zeros(ds[s].logdet, n_obs_nodes, owned), "alloc logdet");
    ST_CUDA(dev_zeros(ds[s].llcomp, n_obs_nodes, owned), "alloc llcomp");
  }
  ST_CUDA(dev_zeros(d_w, n_all, owned), "alloc w");
  ST_CUDA(dev_zeros(d_z, n_all + 1, owned), "alloc z");
  ST_CUDA(dev_upload(xb, d_xb, owned), "upload xb");
  ST_CUDA(dev_zeros(d_V, v_total, owned), "alloc V");
  ST_CUDA(dev_zeros(d_U, u_total, owned), "alloc U");
  ST_CUDA(dev_zeros(d_S, s_total, owned), "alloc S");
  ST_CUDA(dev_zeros(d_Hpred, gpred_total, owned), "alloc Hpred");
  ST_CUDA(dev_zeros(d_sdpred, sd_total_, owned), "alloc sdpred");
  if (probes) {
    ST_CUDA(dev_zeros(d_probe_sig, ri_total, owned), "alloc probe");
    ST_CUDA(dev_zeros(d_probe_smu, n_all, owned), "alloc probe");
  }
  ST_CUDA(dev_zeros(d_scalars, 64 + kMaxStats + 1024, owned), "alloc scalars");
  rowstat_blocks_ = (int)std::min<int64_t>(592, std::max<int64_t>(1, (n_all + 255) / 256));
  ST_CUDA(dev_zeros(d_partial, (long long)rowstat_blocks_ * kMaxStats, owned), "alloc partial");
  ST_CUDA(dev_upload(Bcoeff, d_bcoeff, owned), "upload beta");
  ST_CUDA(dev_upload(tausq_inv, d_tausq_inv, owned), "upload tausq");
  {
    std::vector<int> z1(4, 0);  // [0] BUILD / Gibbs failures (consumed and cleared by the reduction), [1] prediction BUILD
    ST_CUDA(dev_upload(z1, d_fail, owned), "alloc fail");
  }
  ST_CUDA(cudaMallocHost((void**)&h_scalars, (64 + kMaxStats + 1024) * sizeof(double)), "pinned scalars");
  // chain state in device memory (st_chain.hpp) and its pinned host mirror
  {
    void* dc = nullptr;
    ST_CUDA(cudaMalloc(&dc, sizeof(ChainDev)), "alloc chain");
    owned.push_back(dc);
    d_mc = (ChainDev*)dc;
    ST_CUDA(cudaMallocHost((void**)&h_mc, sizeof(ChainDev)), "pinned chain");
    std::memset(h_mc, 0, sizeof(ChainDev));
    h_mc->cur = cur; h_mc->npar = (int)theta[0].size(); h_mc->p = p; h_mc->q = q;
    for (int sl = 0; sl < 2; sl++) {
      std::copy(theta[sl].begin(), theta[sl].end(), h_mc->theta[sl]);
      std::string e2;
      if (!make_covtab(theta[sl].data(), (int)theta[sl].size(), q, h_mc->tab[sl], e2)) { err = e2; return 1; }
    }
    ST_CUDA(cudaMemcpy(d_mc, h_mc, sizeof(ChainDev), cudaMemcpyHostToDevice), "upload chain");
    dslots.s[0] = ds[0]; dslots.s[1] = ds[1]; dslots.chain = d_mc;
  }
  {  // row keys of the device random streams: the row's id in the whole problem (boundary order), node-major here
    std::vector<long long> key(n_all);
    const bool pg = part && !global_rows.empty();
    for (int64_t i = 0; i < n_all; i++) key[i] = pg ? (long long)global_rows[perm[i]] : (long long)perm[i];
    ST_CUDA(dev_upload(key, d_rowkey, owned), "upload rowkey");
    std::vector<long long> ip(iperm.begin(), iperm.end());
    ST_CUDA(dev_upload(ip, d_iperm, owned), "upload iperm");  // (un-permutes the saved rows)
  }
  ST_CUDA(dev_zeros(d_red_scratch, 2 * kReduceScratch, owned), "alloc reduce scratch");  // one set per stream
  ST_CUDA(dev_zeros(d_vrow, n_all, owned), "alloc vrow");
  ST_CUDA(dev_zeros(d_xtx, (long long)q * p * p, owned), "alloc xtx");
  ST_CUDA(dev_zeros(d_bscratch, (long long)q * (3 * p * p + 4 * p) + 8, owned), "alloc beta scratch");  // tausq_beta_kernel's layout
  if (!part) {  // (partitioned handles: after the sums over the ranks, partition_reduce_constants)
    const int rcx = upload_xtx();
    if (rcx) return rcx;
  }
  ST_CUDA(cudaMallocHost((void**)&h_stage, std::max<int64_t>(n_all, 1) * sizeof(double)), "pinned stage");
  // index used by the beta step (SURVEY App. D #12)
  beta_widx_faithful.assign(n_all, -1);
  beta_widx_plain.assign(n_all, -1);
  for (int64_t s = 0; s < n_obs; s++) {
    const int64_t i = iperm[na_ix_all[s]];
    if (part && rank > 0 && i < n_top_rows) continue;  // replicated rows are counted by rank 0 only
    beta_widx_faithful[i] = (int)iperm[s];
    beta_widx_plain[i] = (int)i;
  }
  {
    std::vector<int> tmp(n_all, -1);
    ST_CUDA(dev_upload(tmp, d_obs_widx, owned), "alloc widx");
  }
  beta_widx_mode = -1;
  return 0;
}

int Model::partition_reduce_constants(std::string& e) {
  int rc = 0;
    // XtX and the per-outcome counts are sums over ALL observed rows of the problem: replicated rows once, then all-reduce
    const int nx = q * p * p + q;
    if (nx > 1024) { e = "partition: q*p*p too large"; return 4; }
    for (auto& M : XtX) std::fill(M.a.begin(), M.a.end(), 0.0);
    std::fill(nobs_by_q.begin(), nobs_by_q.end(), 0);
    for (int64_t b : na_ix_all) {
      if (rank > 0 && iperm[b] < n_top_rows) continue;
      const int j = (int)mv_id[b] - 1;
      nobs_by_q[j]++;
      for (int a = 0; a < p; a++)
        for (int c = 0; c < p; c++) XtX[j](a, c) += X[b + (size_t)a * n_all] * X[b + (size_t)c * n_all];
    }
    double* hb = h_scalars + 64 + kMaxStats;
    for (int j = 0; j < q; j++) {
      std::copy(XtX[j].a.begin(), XtX[j].a.end(), hb + (size_t)j * p * p);
      hb[q * p * p + j] = (double)nobs_by_q[j];
    }
    double* db = d_scalars + 64 + kMaxStats;
    ST_CUDA(cudaMemcpyAsync(db, hb, nx * sizeof(double), cudaMemcpyHostToDevice, stream), "H2D XtX");
    rc = allreduce_dev(db, nx);
    if (rc) { e = err; return rc; }
    ST_CUDA(cudaMemcpyAsync(hb, db, nx * sizeof(double), cudaMemcpyDeviceToHost, stream), "D2H XtX");
    ST_CUDA(cudaStreamSynchronize(stream), "sync");
    for (int j = 0; j < q; j++) {
      std::copy(hb + (size_t)j * p * p, hb + (size_t)(j + 1) * p * p, XtX[j].a.begin());
      nobs_by_q[j] = (int64_t)std::llround(hb[q * p * p + j]);
    }
  xtx_pending_ = false;
  return upload_xtx();
}

// XtX and the per-outcome counts of the whole problem to the device (the device-resident beta / tausq steps read them)
int Model::upload_xtx() {
  dvec flat((size_t)q * p * p);
  for (int j = 0; j < q; j++) std::copy(XtX[j].a.begin(), XtX[j].a.end(), flat.begin() + (size_t)j * p * p);
  ST_CUDA(cudaMemcpy(d_xtx, flat.data(), flat.size() * sizeof(double), cudaMemcpyHostToDevice), "upload XtX");
  double nb[kMaxQ] = {0};
  for (int j = 0; j < q; j++) nb[j] = (double)nobs_by_q[j];
  ST_CUDA(cudaMemcpy(d_mc->nobs, nb, sizeof(nb), cudaMemcpyHostToDevice), "upload nobs");
  return 0;
}

int Model::init(std::string& e) {
  // development overrides of the BUILD tiling
  if (const char* v = getenv("ST_BUILD_NS")) force_build_ns = atoi(v);
  if (const char* v = getenv("ST_DEFER")) defer_leaves = atoi(v) != 0;
  if (const char* v = getenv("ST_PDL")) use_pdl = atoi(v) != 0;
  if (const char* v = getenv("ST_OVERLAP")) overlap = atoi(v) != 0;
  if (const char* v = getenv("ST_LLW_OVERLAP")) llw_overlap = atoi(v) != 0;
  if (const char* v = getenv("ST_MAX_COLS")) max_group_cols = atoi(v);
  if (const char* v = getenv("ST_SMEM_BUDGET")) smem_budget = (size_t)atol(v);
  // the Sigi_tot / Smu_tot probes of the Gibbs sweep (st_get_node_state) exist for the parity tests: like H they are kept only
  // on handles created with keep_H (the production / bench configuration writes neither)
  probes = keep_H;
  if (device >= 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && v > 0) n_sm = v;
    else (void)cudaGetLastError();
  }
  if (spread_ctas < 0) spread_ctas = n_sm;
  if (const char* v = getenv("ST_SPREAD")) spread_ctas = atoi(v);
  int rc = build_bookkeeping(e);
  if (rc) return rc;
  if (q * (p + 1) > kMaxStats) { e = "q*(p+1) exceeds 40"; return 4; }
  rc = build_layout(e);
  if (rc) return rc;
  if (n_all >= (1LL << 31)) { e = "n_all must be below 2^31"; return 4; }
  if (device < 0) return 0;  // host-only handle: bookkeeping and layout, no device state (st_get_index only)
  rc = upload(e);
  if (rc) { e = err; return rc; }
  if (part && allreduce_fn) {
    rc = partition_reduce_constants(e);
    if (rc) return rc;
  } else if (part) {
    xtx_pending_ = true;  // no callback: summed when the native communicator is attached (st_attach_nccl)
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------------ operations
int Model::nccl_unique_id(unsigned char* out128, std::string& e) {
  NcclApi& N = nccl();
  if (!N.ok) { e = N.why; return 4; }
  NcclApi::UniqueId id;
  const int rc = N.GetUniqueId(&id);
  if (rc != 0) { e = std::string("ncclGetUniqueId: ") + (N.GetErrorString ? N.GetErrorString(rc) : "error"); return 2; }
  std::memcpy(out128, id.internal, 128);
  return 0;
}

int Model::attach_nccl(const unsigned char* id128) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  if (!part || nranks <= 1) return 0;
  NcclApi& N = nccl();
  if (!N.ok) { err = N.why; return 4; }
  ST_CUDA(cudaSetDevice(device), "cudaSetDevice");
  NcclApi::UniqueId id;
  std::memcpy(id.internal, id128, 128);
  void* comm = nullptr;
  const int rc = N.CommInitRank(&comm, nranks, id, rank);
  if (rc != 0) { err = std::string("ncclCommInitRank: ") + (N.GetErrorString ? N.GetErrorString(rc) : "error"); return 2; }
  nccl_comm = comm;
  if (xtx_pending_) {
    std::string e;
    const int rc2 = partition_reduce_constants(e);
    if (rc2) { if (!e.empty()) err = e; return rc2; }
  }
  return 0;
}

int Model::allreduce_dev(double* dptr, int64_t n) {
  if (!part || nranks <= 1 || n <= 0) return 0;
  if (nccl_comm) {  // in order on the handle's stream: no host synchronisation
    const int rc = nccl().AllReduce(dptr, dptr, (size_t)n, kNcclDouble, kNcclSum, nccl_comm, stream);
    if (rc != 0) { err = std::string("ncclAllReduce: ") + (nccl().GetErrorString ? nccl().GetErrorString(rc) : "error"); return 2; }
    return 0;
  }
  if (!allreduce_fn) { err = "partition: no collective path (call st_attach_nccl or supply st_partition.allreduce)"; return 1; }
  ST_CUDA(cudaStreamSynchronize(stream), "sync before allreduce");
  if (allreduce_fn(allreduce_ctx, dptr, n) != 0) { err = "partition: the allreduce callback failed"; return 1; }
  return 0;
}

// sum of the per-block log-density pieces (:987-988 / :815-816) of the slot `rel` into dev_red8 (device): [0..2] the
// replicated blocks (or nothing), [4..6] the rest, all-reduced over the ranks of a partition; [6] = failed factorisations.
// out3_host (host-driven path) = {loglik_w, logdetCi, failures}: one D2H + synchronisation.
int Model::reduce_loglik(int rel, int* fail, double* dev_red8, double* out3_host) {
  ST_CUDA(launch_loglik_reduce(dslots, rel, part ? n_top_slots : 0, n_obs_nodes, fail, dev_red8, d_red_scratch, stream), "loglik_reduce");
  n_launches++;
  if (part) { int rc = allreduce_dev(dev_red8 + 4, 3); if (rc) return rc; }
  if (!out3_host) return 0;
  ST_CUDA(cudaMemcpyAsync(h_scalars, dev_red8, 8 * sizeof(double), cudaMemcpyDeviceToHost, stream), "D2H scalars");
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  out3_host[0] = h_scalars[0] + h_scalars[4];
  out3_host[1] = h_scalars[1] + h_scalars[5];
  out3_host[2] = h_scalars[6];
  return 0;
}

int Model::theta_update(int slot, const double* th) {
  dvec& t = theta[phys(slot)];
  std::copy(th, th + t.size(), t.begin());
  return 0;
}

int Model::push_slot_theta(int ps) {
  ThetaPack pk;
  std::string e;
  pk.n = (int)theta[ps].size();
  if (pk.n > kMaxPar) { err = "more than 64 covariance parameters"; return 4; }
  std::copy(theta[ps].begin(), theta[ps].end(), pk.theta);
  if (!make_covtab(theta[ps].data(), pk.n, q, pk.tab, e)) { err = e; return 1; }
  ST_CUDA(launch_chain_set_theta(d_mc, ps == cur ? 0 : 1, pk, stream), "chain_set_theta_kernel");
  return 0;
}

// levels [l0, l1) of a BUILD of the slot `rel` on stream `st`; no_density: their log-density pieces are left to an LLW pass
int Model::launch_build_levels(int rel, int l0, int l1, bool no_density, cudaStream_t st) {
  NvtxRange nvtx(no_density ? "BUILD (upper levels, second stream)" : "BUILD");
  // ST_PROFILE_BUILD=1: per-phase clock64() totals of build_level_kernel, printed per level (development aid)
  static const bool profile = getenv("ST_PROFILE_BUILD") != nullptr;
  unsigned long long* d_prof = nullptr;
  if (profile) {
    cudaMalloc((void**)&d_prof, 16 * sizeof(unsigned long long));
  }
  bool first_launch = true;
  if (l1 < 0) l1 = (int)levels.size();
  if (!st) st = stream;
  for (int li = l0; li < l1; li++) {
    auto& L = levels[li];
    for (const auto& B : L.build_launches) {
      cudaEvent_t pe0 = nullptr, pe1 = nullptr;
      if (profile) {
        cudaMemsetAsync(d_prof, 0, 16 * sizeof(unsigned long long), st);
        cudaEventCreate(&pe0); cudaEventCreate(&pe1);
        cudaEventRecord(pe0, st);
      }
      // every launch but the first of a BUILD may start before its predecessor has drained (programmatic dependent
      // launch): it waits inside the kernel before it reads the ancestors' row blocks
      ST_CUDA(launch_build(L.is_ref ? 0 : 1, dt, dslots, rel, nullptr, nullptr, keep_H ? 1 : 0, d_grp_slot0 + B.grp0, d_grp_nn + B.grp0,
                           B.ngrp, d_w, d_fail, B.ns, (L.deferrable ? 1 : 0) | (no_density ? 4 : 0), B.smem, st, B.threads, d_prof,
                           use_pdl && !first_launch && !profile),
              "build_level_kernel");
      first_launch = false;
      n_launches++;
      if (profile) {
        unsigned long long h[16];
        cudaEventRecord(pe1, st);
        cudaStreamSynchronize(st);
        float pms = 0;
        cudaEventElapsedTime(&pms, pe0, pe1);
        cudaEventDestroy(pe0); cudaEventDestroy(pe1);
        cudaMemcpy(h, d_prof, sizeof(h), cudaMemcpyDeviceToHost);
        double tot = 0;
        for (int i = 0; i < 7; i++) tot += (double)h[i];
        fprintf(stderr, "[build profile] level slot0=%d groups=%d ref=%d threads=%d ns=%d smem=%zu  %.3f ms  cycles/group=%.0f : setup %.1f%% cov %.1f%% fwd %.1f%% ZtZ %.1f%% chol %.1f%% Y %.1f%% bwd+out %.1f%%\n",
                L.slot0, B.ngrp, L.is_ref, B.threads, B.ns, B.smem, pms, tot / std::max(1, B.ngrp), 100 * h[0] / tot, 100 * h[1] / tot,
                100 * h[2] / tot, 100 * h[3] / tot, 100 * h[4] / tot, 100 * h[5] / tot, 100 * h[6] / tot);
        if (L.is_ref) fprintf(stderr, "      chol (warp pair 0: factorise + invert, one pivot apart): %.1f%% of kernel\n", 100 * h[8] / tot);
      }
    }
  }
  if (profile) cudaFree(d_prof);
  return 0;
}

// The deferred half of BUILD: childless non-reference blocks of the slot `rel` get their G (backward sweep over the parked
// Z).  run_flag (device-resident chain): a device int, the launches are no-ops when it is 0.
int Model::launch_deferred_half(int rel, const int* run_flag, cudaStream_t st) {
  NvtxRange nvtx("BUILD deferred half");
  if (!st) st = stream;
  for (auto& L : levels) {
    if (!L.deferrable) continue;
    for (const auto& B : L.build_launches) {
      ST_CUDA(launch_build(1, dt, dslots, rel, nullptr, nullptr, 0, d_grp_slot0 + B.grp0, d_grp_nn + B.grp0, B.ngrp, d_w, d_fail, B.ns, 2,
                           B.smem, st, B.threads, nullptr, false, run_flag),
              "build_level_kernel(deferred half)");
      n_launches++;
    }
  }
  return 0;
}
int Model::complete_slot(int pslot) {
  if (!deferred_[pslot]) return 0;
  const int rc = launch_deferred_half(pslot == cur ? 0 : 1, nullptr, stream);
  if (rc) return rc;
  deferred_[pslot] = false;
  return 0;
}

int Model::get_loglik_comps_w(int slot, double* out3) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  const int ps = phys(slot);
  int rc = push_slot_theta(ps);
  if (rc) return rc;
  ST_CUDA(cudaMemsetAsync(d_fail, 0, sizeof(int), stream), "memset");
  rc = launch_build_levels(ps == cur ? 0 : 1, 0, -1, false, stream);
  if (rc) return rc;
  for (auto& L : levels) if (L.deferrable) deferred_[ps] = true;
  double r3[3];
  rc = reduce_loglik(ps == cur ? 0 : 1, d_fail, d_mc->red_build, r3);
  if (rc) return rc;
  const bool ok = r3[2] == 0.0;
  if (ok) { loglik_w[ps] = r3[0]; logdetCi[ps] = r3[1]; }  // on failure the reference leaves them untouched (:971-982)
  if (ps == cur) { gram_stale = true; pred_H_valid = false; }
  else alter_scratch = false;
  out3[0] = loglik_w[ps]; out3[1] = logdetCi[ps]; out3[2] = ok ? 1.0 : 0.0;
  return 0;
}

int Model::upload_rows(const double* boundary_order, double* dev) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  for (int64_t i = 0; i < n_all; i++) h_stage[i] = boundary_order[perm[i]];
  ST_CUDA(cudaMemcpyAsync(dev, h_stage, n_all * sizeof(double), cudaMemcpyHostToDevice, stream), "H2D rows");
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  return 0;
}

int Model::draw_normals(uint64_t seed) {
  ST_CUDA(launch_normals(d_z, n_all, seed, sweep_counter++, d_rowkey, nullptr, stream), "normals_kernel");
  n_launches++;
  return 0;
}

int Model::refresh_grams(const int* run_flag, cudaStream_t st) {
  NvtxRange nvtx("Gram refresh");
  if (!st || part) st = stream;  // (a partitioned handle's collective stays on the main stream)
  if (!run_flag) { int rc = complete_slot(cur); if (rc) return rc; }
  bool chained = false;  // the previous launch on the stream is a gram level: programmatic dependent launch is safe
  for (int g = (int)levels.size() - 1; g >= 0; g--) {
    if (part && n_top_levels >= 1 && g == n_top_levels - 1) {  // children of this level live on several ranks
      // (unconditional also in the device-resident chain: every rank must enter the collective, and summing the unchanged
      // tiles again gives the same pseudo-child)
      ST_CUDA(launch_frontier_sum(dt, (int)h_front_pseudo.size(), d_front_pseudo, d_front_c0, d_front_c1, d_front_vlen, d_front_ulen,
                                  d_V, d_U, 0, 1, stream), "frontier_sum_kernel");
      n_launches++;
      int rc = allreduce_dev(d_U + u_front0, u_front_len);
      if (rc) return rc;
      chained = false;
    }
    if (levels[g].gram_skip) continue;  // all blocks of the level are fused into their parents
    static const bool profile = getenv("ST_PROFILE_GIBBS") != nullptr;
    cudaEvent_t pe0 = nullptr, pe1 = nullptr;
    if (profile) { cudaEventCreate(&pe0); cudaEventCreate(&pe1); cudaEventRecord(pe0, st); }
    ST_CUDA(launch_gram(dt, dslots, levels[g].slot0, levels[g].nslots, d_U, d_S, levels[g].gram_rch, levels[g].gram_ldx, levels[g].gram_tiles,
                        levels[g].gram_stage_off, levels[g].gram_threads, st, run_flag, use_pdl && !profile && chained),
            "gram_level_kernel");
    chained = true;
    n_launches++;
    if (profile) {
      cudaEventRecord(pe1, st);
      cudaStreamSynchronize(st);
      float pms = 0;
      cudaEventElapsedTime(&pms, pe0, pe1);
      cudaEventDestroy(pe0); cudaEventDestroy(pe1);
      fprintf(stderr, "[gram profile] level slot0=%d nodes=%d rch=%d ldx=%d  %.3f ms\n", levels[g].slot0, levels[g].nslots,
              levels[g].gram_rch, levels[g].gram_ldx, pms);
    }
  }
  if (!run_flag) gram_stale = false;
  return 0;
}

// the level launches of one Gibbs sweep, leaves to root; fail_ptr: device int that counts failed factorisations; iloo: the
// sweep also forms the integrated log-likelihood into d_ll_int_
int Model::gibbs_launch_only(int* fail_ptr, bool iloo) {
  NvtxRange nvtx("GIBBS");
  for (int g = (int)levels.size() - 1; g >= 0; g--) {
    const LevelInfo& L = levels[g];
    if (part && n_top_levels >= 1 && g == n_top_levels - 1) {
      ST_CUDA(launch_frontier_sum(dt, (int)h_front_pseudo.size(), d_front_pseudo, d_front_c0, d_front_c1, d_front_vlen, d_front_ulen,
                                  d_V, d_U, 1, 0, stream), "frontier_sum_kernel");
      n_launches++;
      int rc = allreduce_dev(d_V + v_front0, v_front_len);
      if (rc) return rc;
    }
    static const bool profile = getenv("ST_PROFILE_GIBBS") != nullptr;  // development aid: per-level event timing
    cudaEvent_t pe0 = nullptr, pe1 = nullptr;
    if (profile) { cudaEventCreate(&pe0); cudaEventCreate(&pe1); cudaEventRecord(pe0, stream); }
    ST_CUDA(launch_gibbs(L.is_ref, dt, dslots, L.slot0, L.nslots, d_w, d_xb, d_z, d_tausq_inv, d_S, d_V,
                         probes ? d_probe_sig : nullptr, probes ? d_probe_smu : nullptr, fail_ptr, L.smem_gibbs, stream,
                         use_pdl && !profile && g != (int)levels.size() - 1, iloo ? d_ll_int_ : nullptr,
                         iloo ? d_ll_int_ + n_all : nullptr),
            "gibbs_level_kernel");
    n_launches++;
    if (profile) {
      cudaEventRecord(pe1, stream);
      cudaStreamSynchronize(stream);
      float pms = 0;
      cudaEventElapsedTime(&pms, pe0, pe1);
      cudaEventDestroy(pe0); cudaEventDestroy(pe1);
      fprintf(stderr, "[gibbs profile] level slot0=%d nodes=%d ref=%d smem=%zu maxm=%d maxP=%d  %.3f ms\n", L.slot0, L.nslots, L.is_ref,
              L.smem_gibbs, L.maxm, L.maxP, pms);
    }
  }
  return 0;
}

int Model::deal_with_w(const double* z, uint64_t seed) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  if (z) { int rc = upload_rows(z, d_z); if (rc) return rc; }
  else { int rc = draw_normals(seed); if (rc) return rc; }
  stats_valid_mode_ = -1;  // w is about to change
  { int rc = complete_slot(cur); if (rc) return rc; }
  if (gram_stale) { int rc = refresh_grams(); if (rc) return rc; }
  const bool iloo = (keep_mask & ST_KEEP_LOGLIK_INT) != 0;
  if (iloo) { int rc = alloc_loglik_int(); if (rc) return rc; }
  ST_CUDA(cudaMemsetAsync(d_fail, 0, sizeof(int), stream), "memset");
  int rc = gibbs_launch_only(d_fail, iloo);
  if (rc) return rc;
  // failed factorisations, agreed over the ranks of a partition (every rank must take the same exit): the count rides in an
  // 8-double reduction slot, all-reduced on the stream
  double* slot8 = d_scalars + 48;
  ST_CUDA(launch_loglik_reduce(dslots, 0, 0, 0, d_fail, slot8, d_red_scratch, stream), "fail count");
  if (part) { rc = allreduce_dev(slot8 + 4, 3); if (rc) return rc; }
  ST_CUDA(cudaMemcpyAsync(h_scalars + 48, slot8, 8 * sizeof(double), cudaMemcpyDeviceToHost, stream), "D2H fail");
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  if (h_scalars[48 + 6] != 0.0) { err = "Error at gibbs_sample_w: conditional precision not positive definite"; return 3; }
  if (iloo) ll_int_valid_ = true;
  return 0;
}

int Model::alloc_loglik_int() {
  if (d_ll_int_) return 0;
  ST_CUDA(dev_zeros(d_ll_int_, 2 * n_all, owned), "alloc integrated log-likelihood");
  ST_CUDA(cudaMemsetAsync(d_ll_int_, 0xff, n_all * sizeof(double), stream), "memset");  // (all bits set: a NaN)
  const double nan = std::numeric_limits<double>::quiet_NaN();
  for (int64_t i = 0; i < n_all; i++) h_stage[i] = std::isfinite(y[perm[i]]) ? y[perm[i]] : nan;
  ST_CUDA(cudaMemcpyAsync(d_ll_int_ + n_all, h_stage, n_all * sizeof(double), cudaMemcpyHostToDevice, stream), "H2D y");
  ST_CUDA(cudaStreamSynchronize(stream), "sync");  // (h_stage is free again)
  return 0;
}

int Model::get_loglik_int(double* out) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  if (!ll_int_valid_) {
    err = "st_get_loglik_int: no sweep has formed the integrated log-likelihood (st_keep_samples_on_device with ST_KEEP_LOGLIK_INT "
          "before st_deal_with_w or st_mcmc_run)";
    return 1;
  }
  ST_CUDA(cudaMemcpyAsync(h_stage, d_ll_int_, n_all * sizeof(double), cudaMemcpyDeviceToHost, stream), "D2H integrated log-likelihood");
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  for (int64_t i = 0; i < n_all; i++) out[perm[i]] = h_stage[i];
  return 0;
}

int Model::get_loglik_w(int slot, double* out2) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  const int ps = phys(slot);
  if (ps != cur && alter_scratch) { err = "the alter slot holds a BUILD of st_predict_new: st_get_loglik_comps_w(h, 1, ...) rebuilds it first"; return 1; }
  { int rc = complete_slot(ps); if (rc) return rc; }
  ST_CUDA(launch_llw(dt, dslots, ps == cur ? 0 : 1, 0, n_obs_nodes, d_w, llw_maxlen_, stream), "llw_kernel");
  n_launches++;
  double r3[3];
  int rc = reduce_loglik(ps == cur ? 0 : 1, nullptr, d_mc->red_llw, r3);
  if (rc) return rc;
  loglik_w[ps] = r3[0];
  logdetCi[ps] = r3[1];
  out2[0] = loglik_w[ps]; out2[1] = logdetCi[ps];
  return 0;
}

void Model::accept_make_change() {
  cur = 1 - cur;
  gram_stale = true;
  pred_H_valid = false;
  if (!stream) return;
  if (launch_chain_flip(d_mc, stream) != cudaSuccess) { err = "chain_flip_kernel failed"; return; }
  if (complete_slot(cur) != 0) deferred_[cur] = true;  // (an error here resurfaces at the next consumer)
}

int Model::predict(bool theta_changed) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  if (pred_level.nslots == 0) return 0;
  if (theta_changed || !pred_H_valid) {
    int rc = push_slot_theta(cur);
    if (rc) return rc;
    for (const auto& B : pred_level.build_launches) {
      ST_CUDA(launch_build(2, dt, dslots, 0, d_Hpred, d_sdpred, 0, d_grp_slot0 + B.grp0, d_grp_nn + B.grp0, B.ngrp, d_w, d_fail + 1, B.ns, 0,
                           B.smem, stream, B.threads, nullptr),
              "build_level_kernel(predict)");
      n_launches++;
    }
    pred_H_valid = true;
  }
  stats_valid_mode_ = -1;  // w of the prediction rows changes
  ST_CUDA(launch_predict_sample(dt, pred_level.slot0, pred_level.nslots, d_Hpred, d_sdpred, d_w, d_z, stream), "predict_sample_kernel");
  n_launches++;
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  return 0;
}

// statistics of the beta / tausq steps into d_scalars + 8 (all-reduced over the ranks); no synchronisation
int Model::enqueue_stats() {
  NvtxRange nvtx("tausq / beta statistics");
  ST_CUDA(launch_rowstats(dt, d_obs_widx, n_all, p, q, d_w, d_xb, d_partial, rowstat_blocks_, d_scalars + 8, stream), "rowstats_kernel");
  n_launches += 2;
  return allreduce_dev(d_scalars + 8, q * (p + 1));
}

int Model::rowstats(bool faithful_index) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  const int mode = faithful_index ? 1 : 0;
  // the tausq and the beta step of one iteration read the same statistics (neither w nor XB changes in between)
  if (stats_valid_mode_ == mode) return 0;
  if (beta_widx_mode != mode) {
    const std::vector<int>& src = faithful_index ? beta_widx_faithful : beta_widx_plain;
    ST_CUDA(cudaMemcpyAsync(d_obs_widx, src.data(), n_all * sizeof(int), cudaMemcpyHostToDevice, stream), "H2D widx");
    ST_CUDA(cudaStreamSynchronize(stream), "sync");
    beta_widx_mode = mode;
  }
  int rc = enqueue_stats();
  if (rc) return rc;
  ST_CUDA(cudaMemcpyAsync(h_scalars + 8, d_scalars + 8, q * (p + 1) * sizeof(double), cudaMemcpyDeviceToHost, stream), "D2H stats");
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  stats_valid_mode_ = mode;
  return 0;
}

// gibbs_sample_tausq spamtree_model.cpp:1393-1417
int Model::gibbs_sample_tausq(const double* fixed) {
  if (part && beta_widx_mode == -1) beta_widx_mode = -2;
  int rc = rowstats(part ? false : (beta_widx_mode != 0));
  if (rc) return rc;
  for (int j = 0; j < q; j++) {
    const double bcore = h_scalars[8 + j * (p + 1) + p];
    const double aparam = 2.01 + nobs_by_q[j] / 2.0;
    const double bparam = 1.0 / (1.0 + .5 * bcore);
    tausq_inv[j] = fixed ? fixed[j] : rng.gamma(aparam, bparam);
  }
  ST_CUDA(cudaMemcpyAsync(d_tausq_inv, tausq_inv.data(), q * sizeof(double), cudaMemcpyHostToDevice, stream), "H2D tausq");
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  return 0;
}

// gibbs_sample_beta spamtree_model.cpp:1364-1391
int Model::gibbs_sample_beta(const double* zb, bool faithful_index) {
  if (part && faithful_index) {
    err = "partitioned runs support only the corrected beta row index (faithful_index = 0): the reference's mis-indexing "
          "(SURVEY App. D #12) mixes rows that live on different ranks";
    return 4;
  }
  int rc = rowstats(faithful_index);
  if (rc) return rc;
  for (int j = 0; j < q; j++) {
    SmallMat Si(p);
    for (int a = 0; a < p; a++)
      for (int b = 0; b < p; b++) Si(a, b) = tausq_inv[j] * XtX[j](a, b) + (a == b ? .01 : 0.0);  // Vi = .01 I (:157)
    for (int a = 0; a < p; a++)
      for (int b = 0; b < a; b++) Si(a, b) = Si(b, a);  // symmatu
    if (!small_chol(Si)) { err = "beta step: precision not positive definite"; return 3; }
    SmallMat Sc = small_inv_lower(Si);
    dvec xp(p), t(p, 0.0), bmu(p, 0.0), zz(p), sz(p, 0.0);
    for (int a = 0; a < p; a++) xp[a] = 0.0 + tausq_inv[j] * h_scalars[8 + j * (p + 1) + a];  // Vim = 0 (:158-159)
    for (int a = 0; a < p; a++)
      for (int b = 0; b <= a; b++) t[a] += Sc(a, b) * xp[b];
    for (int a = 0; a < p; a++)
      for (int b = a; b < p; b++) bmu[a] += Sc(b, a) * t[b];
    for (int a = 0; a < p; a++) zz[a] = zb ? zb[a + (size_t)j * p] : rng.norm();
    for (int a = 0; a < p; a++)
      for (int b = a; b < p; b++) sz[a] += Sc(b, a) * zz[b];
    for (int a = 0; a < p; a++) Bcoeff[a + (size_t)j * p] = bmu[a] + sz[a];
  }
  ST_CUDA(cudaMemcpyAsync(d_bcoeff, Bcoeff.data(), (size_t)p * q * sizeof(double), cudaMemcpyHostToDevice, stream), "H2D beta");
  stats_valid_mode_ = -1;  // XB changes
  ST_CUDA(launch_xb(dt, n_all, p, d_bcoeff, d_xb, stream), "xb_kernel");
  n_launches++;
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  return 0;
}
int Model::get_w(double* out) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  ST_CUDA(cudaMemcpyAsync(h_stage, d_w, n_all * sizeof(double), cudaMemcpyDeviceToHost, stream), "D2H w");
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  for (int64_t i = 0; i < n_all; i++) out[perm[i]] = h_stage[i];
  return 0;
}
int Model::set_w(const double* in) { stats_valid_mode_ = -1; return upload_rows(in, d_w); }

int Model::save_rows(CopyOut& co, int k, double* dev, double* host) {
  // (a slot of the device store is written once: only a staging slot waits for the copy that read it)
  double* buf = dev ? dev : co.buffer(k);
  if (!buf) return 2;
  if (k == 0) ST_CUDA(launch_permute(d_w, buf, d_iperm, n_all, stream), "permute_kernel");
  else ST_CUDA(launch_yhat(dt, d_w, d_xb, d_tausq_inv, d_iperm, d_rowkey, n_all, d_mc, buf, stream), "yhat_kernel");
  n_launches++;
  const double* src = buf;
  return co.send(k, &host, &src, 1, n_all);
}

int CopyOut::chk(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return 0;
  err_ = std::string("CUDA error in ") + what + ": " + cudaGetErrorString(e);
  return 2;  // ST_ERR_CUDA
}

int CopyOut::open(std::initializer_list<double*> hosts, size_t bytes_each, int nslots, size_t n) {
  n_ = n;
  copied_.assign(nslots, nullptr);
  pending_.assign(nslots, 0);
  if (int rc = chk(cudaMalloc((void**)&staging_, std::max<size_t>(nslots * n, 1) * sizeof(double)), "alloc staging")) {
    staging_ = nullptr;
    return rc;
  }
  if (int rc = chk(cudaEventCreateWithFlags(&ready_, cudaEventDisableTiming), "cudaEventCreate")) return rc;
  for (cudaEvent_t& e : copied_)
    if (int rc = chk(cudaEventCreateWithFlags(&e, cudaEventDisableTiming), "cudaEventCreate")) return rc;
  for (double* h : hosts) {
    if (!h || bytes_each == 0) continue;
    if (cudaHostRegister(h, bytes_each, cudaHostRegisterPortable) == cudaSuccess) locked_.push_back(h);
    else (void)cudaGetLastError();  // (the copies still go there, see the class comment)
  }
  return 0;
}

double* CopyOut::buffer(int slot) {
  if (pending_[slot] && chk(cudaStreamWaitEvent(st_, copied_[slot], 0), "wait for the copy of an earlier row")) return nullptr;
  return staging_ + (size_t)slot * n_;
}

int CopyOut::send(int slot, double* const* dst, const double* const* src, int count, size_t n) {
  if (std::none_of(dst, dst + count, [](double* d) { return d != nullptr; })) return 0;
  if (int rc = chk(cudaEventRecord(ready_, st_), "event")) return rc;
  if (int rc = chk(cudaStreamWaitEvent(cs_, ready_, 0), "wait")) return rc;
  for (int c = 0; c < count; c++)
    if (dst[c])
      if (int rc = chk(cudaMemcpyAsync(dst[c], src[c], n * sizeof(double), cudaMemcpyDeviceToHost, cs_), "D2H rows")) return rc;
  if (int rc = chk(cudaEventRecord(copied_[slot], cs_), "event")) return rc;
  pending_[slot] = 1;
  return 0;
}

int CopyOut::finish() {
  if (!staging_) return 0;
  std::fill(pending_.begin(), pending_.end(), 0);
  return chk(cudaStreamSynchronize(cs_), "sync of the copies");
}

CopyOut::~CopyOut() {
  if (staging_) {  // (an early exit may leave kernels that write the staging, or copies from it, in flight)
    cudaStreamSynchronize(cs_);
    cudaStreamSynchronize(st_);
  }
  for (void* p : locked_) cudaHostUnregister(p);
  for (cudaEvent_t e : copied_) if (e) cudaEventDestroy(e);
  if (ready_) cudaEventDestroy(ready_);
  if (staging_) cudaFree(staging_);
}

int Model::get_xb(double* out) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  ST_CUDA(cudaMemcpyAsync(h_stage, d_xb, n_all * sizeof(double), cudaMemcpyDeviceToHost, stream), "D2H xb");
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  for (int64_t i = 0; i < n_all; i++) out[perm[i]] = h_stage[i];
  return 0;
}
int Model::set_tausq_inv(const double* t) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  std::copy(t, t + q, tausq_inv.begin());
  ST_CUDA(cudaMemcpyAsync(d_tausq_inv, tausq_inv.data(), q * sizeof(double), cudaMemcpyHostToDevice, stream), "H2D tausq");
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  return 0;
}
int Model::sync() {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  return 0;
}

int Model::get_node_state(int slot, int u, const std::string& which, double* out, int64_t cap, int64_t* count) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  const int ps = phys(slot);
  { int rc = complete_slot(ps); if (rc) return rc; }
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  auto emit = [&](const dvec& v) {
    *count = (int64_t)v.size();
    if (out) for (int64_t i = 0; i < (int64_t)v.size() && i < cap; i++) out[i] = v[i];
    return 0;
  };
  if (which == "logdetCi_comps" || which == "loglik_w_comps") {
    dvec d(n_obs_nodes), o(n_blocks, 0.0);
    ST_CUDA(cudaMemcpy(d.data(), (which == "logdetCi_comps") ? ds[ps].logdet : ds[ps].llcomp, n_obs_nodes * sizeof(double), cudaMemcpyDeviceToHost), "D2H comps");
    for (int s = 0; s < n_obs_nodes; s++) o[block_of_slot[s]] = d[s];
    return emit(o);
  }
  if (u < 0 || u >= n_blocks) { err = "block id out of range"; return 1; }
  const int s = slot_of_block[u];
  const bool pred = s >= n_obs_nodes;
  const int m = h_m[s], P = h_P[s];
  if (which == "H" || which == "G") {
    const double* src = nullptr;
    if (pred) { if (which == "G") { err = "prediction blocks have no G"; return 1; } src = d_Hpred; }
    else if (which == "G") src = ds[ps].G;
    else { if (!keep_H) { err = "H was not kept (keep_H = 0)"; return 1; } src = ds[ps].H; }
    const int gs = h_gs[s];
    const long long tot = (long long)m * gs;
    dvec t(std::max<long long>(tot, 1)), o((size_t)m * P);
    if (tot) ST_CUDA(cudaMemcpy(t.data(), src + h_goff[s], tot * sizeof(double), cudaMemcpyDeviceToHost), "D2H H");
    for (int r = 0; r < m; r++)
      for (int pp = 0; pp < P; pp++) o[r + (size_t)pp * m] = t[(size_t)r * gs + pp];
    return emit(o);
  }
  if (which == "Ri") {
    if (pred) {
      dvec o(m);
      ST_CUDA(cudaMemcpy(o.data(), d_sdpred + h_rioff[s], m * sizeof(double), cudaMemcpyDeviceToHost), "D2H sd");
      return emit(o);
    }
    if (isref_host_[s]) {
      const int rsm = tile_rs(m);
      dvec t((size_t)m * rsm), o((size_t)m * m);
      ST_CUDA(cudaMemcpy(t.data(), ds[ps].Ri + h_rioff[s], t.size() * sizeof(double), cudaMemcpyDeviceToHost), "D2H Ri");
      for (int r = 0; r < m; r++)
        for (int c = 0; c < m; c++) o[r + (size_t)c * m] = t[(size_t)r * rsm + c];
      return emit(o);
    }
    dvec o(m);
    ST_CUDA(cudaMemcpy(o.data(), ds[ps].Ri + h_rioff[s], m * sizeof(double), cudaMemcpyDeviceToHost), "D2H ri");
    return emit(o);
  }
  if (which == "Sigi_tot" || which == "Smu_tot") {
    if (pred || !probes) { err = "no Gibbs probe for this block (prediction block or probes disabled)"; return 1; }
    if (which == "Smu_tot") {
      dvec o(m);
      ST_CUDA(cudaMemcpy(o.data(), d_probe_smu + h_row0[s], m * sizeof(double), cudaMemcpyDeviceToHost), "D2H smu");
      return emit(o);
    }
    const size_t n = isref_host_[s] ? (size_t)m * m : (size_t)m;
    dvec o(n);
    ST_CUDA(cudaMemcpy(o.data(), d_probe_sig + h_rioff[s], n * sizeof(double), cudaMemcpyDeviceToHost), "D2H sig");
    return emit(o);
  }
  err = "unknown state name: " + which;
  return 1;
}

int Model::get_index(const std::string& which, int u, int c, int64_t* out, int64_t cap, int64_t* count) {
  ivec r;
  auto emit = [&](const ivec& v) {
    *count = (int64_t)v.size();
    if (out) for (int64_t i = 0; i < (int64_t)v.size() && i < cap; i++) out[i] = v[i];
    return 0;
  };
  if (which == "blocks_not_empty") return emit(blocks_not_empty);
  if (which == "blocks_predicting") return emit(blocks_predicting);
  if (which == "block_is_reference") return emit(block_is_reference);
  if (which == "block_ct_obs") return emit(block_ct_obs);
  if (which == "n_actual_groups") { r.push_back(n_actual_groups); return emit(r); }
  if (which == "u_by_block_groups") {
    if (u < 0 || u >= n_actual_groups) { err = "group out of range"; return 1; }
    return emit(u_by_block_groups[u]);
  }
  if (which == "build_plan") {
    // The launch plan chosen at creation (host-only handles too), for tests that must know which kernel paths a tree reaches.
    // [n_launch, n_level], then n_launch records of 9 for the BUILD launches of every observed level and of the prediction
    // level: {level (-1: prediction blocks), mode, groups, ns, threads, dynamic smem bytes, largest nn, largest NCp,
    // largest npair}; then n_level records of 9 for the observed levels: {deferrable, early (BUILD underneath the sweep of
    // a device-resident chain), gram_rch, largest staged rows of a block, gram_stage_off, gram_threads, largest children
    // count, largest nch * ntile, largest Gram item count} (the last five over the blocks gram_level_kernel processes, i.e.
    // not fused)
    ivec lr;
    int nlaunch = 0;
    auto launches = [&](const LevelInfo& L, int lev, int mode) {
      const int xcol = L.deferrable ? 1 : 0;
      for (const auto& B : L.build_launches) {
        long long mnn = 0, mncp = 0, mpair = 0;
        for (int g = B.grp0; g < B.grp0 + B.ngrp; g++) {
          int ncols = xcol;
          for (int d = 0; d < h_grp_nn[g]; d++) ncols += h_m[h_grp_slot0[g] + d];
          const int ncp = (ncols + 7) & ~7;
          mnn = std::max<long long>(mnn, h_grp_nn[g]);
          mncp = std::max<long long>(mncp, ncp);
          mpair = std::max<long long>(mpair, build_npair(ncp >> 3, B.threads / 32));
        }
        r.insert(r.end(), {(int64_t)lev, (int64_t)mode, (int64_t)B.ngrp, (int64_t)B.ns, (int64_t)B.threads, (int64_t)B.smem, mnn, mncp, mpair});
        nlaunch++;
      }
    };
    for (int l = 0; l < (int)levels.size(); l++) {
      const LevelInfo& L = levels[l];
      launches(L, l, L.is_ref ? 0 : 1);
      long long mch = 0, mct = 0;
      for (int t = L.slot0; t < L.slot0 + L.nslots; t++) {
        if (h_ufused[t]) continue;
        const int nch = h_child_ptr[t + 1] - h_child_ptr[t];
        mch = std::max<long long>(mch, nch);
        mct = std::max<long long>(mct, (long long)nch * (h_k[t] + (h_soff[t] >= 0 ? 1 : 0)));
      }
      lr.insert(lr.end(), {(int64_t)L.deferrable, (int64_t)(overlap && l < n_early_levels_), (int64_t)L.gram_rch, (int64_t)L.gram_maxrows,
                           (int64_t)L.gram_stage_off, (int64_t)L.gram_threads, mch, mct, (int64_t)L.gram_maxitems});
    }
    launches(pred_level, -1, 2);
    r.insert(r.begin(), {(int64_t)nlaunch, (int64_t)levels.size()});
    r.insert(r.end(), lr.begin(), lr.end());
    return emit(r);
  }
  if (which == "build_groups") {
    // every BUILD work group in launch order, 6 per group: {level (-1: prediction blocks), first slot, nn, NCp, threads,
    // npair}.  Two handles whose groups agree run the same reductions for every block.
    auto groups = [&](const LevelInfo& L, int lev) {
      const int xcol = L.deferrable ? 1 : 0;
      for (const auto& B : L.build_launches)
        for (int g = B.grp0; g < B.grp0 + B.ngrp; g++) {
          int ncols = xcol;
          for (int d = 0; d < h_grp_nn[g]; d++) ncols += h_m[h_grp_slot0[g] + d];
          const int ncp = (ncols + 7) & ~7;
          r.insert(r.end(), {(int64_t)lev, (int64_t)h_grp_slot0[g], (int64_t)h_grp_nn[g], (int64_t)ncp, (int64_t)B.threads,
                             (int64_t)build_npair(ncp >> 3, B.threads / 32)});
        }
    };
    for (int l = 0; l < (int)levels.size(); l++) groups(levels[l], l);
    groups(pred_level, -1);
    return emit(r);
  }
  if (u < 0 || u >= n_blocks) { err = "block id out of range"; return 1; }
  if (which == "parents_indexing") {  // init_indexing :325-335
    for (int64_t t = parents.ptr[u]; t < parents.ptr[u + 1]; t++) {
      const int64_t pa = parents.idx[t];
      r.insert(r.end(), indexing.row(pa), indexing.row(pa) + indexing.len(pa));
    }
    return emit(r);
  }
  if (which == "children_indexing") {
    for (int64_t t = children.ptr[u]; t < children.ptr[u + 1]; t++) {
      const int64_t chd = children.idx[t];
      r.insert(r.end(), indexing.row(chd), indexing.row(chd) + indexing.len(chd));
    }
    return emit(r);
  }
  auto dim_by_parent = [&](int b) {  // init_finalize :362-373
    ivec d;
    if (indexing.len(b) == 0) return d;
    d.push_back(0);
    for (int64_t t = parents.ptr[b]; t < parents.ptr[b + 1]; t++) d.push_back(d.back() + indexing.len(parents.idx[t]));
    return d;
  };
  if (which == "dim_by_parent") return emit(dim_by_parent(u));
  if (which == "this_is_jth_child") {  // :411-417
    r.assign(parents.len(u), 0);
    if (block_ct_obs[u] > 0)
      for (int64_t t = 0; t < parents.len(u); t++) {
        const int64_t pa = parents.idx[parents.ptr[u] + t];
        const int64_t* b = children.row(pa);
        r[t] = (int64_t)(std::find(b, b + children.len(pa), (int64_t)u) - b);
      }
    return emit(r);
  }
  if (which == "u_is_which_col") {  // :388-409: (firstcol, lastcol) of u inside child c's parent set
    if (c < 0 || c >= children.len(u)) { err = "child position out of range"; return 1; }
    const int child = (int)children.idx[children.ptr[u] + c];
    const int64_t* b = parents.row(child);
    const int64_t wh = std::find(b, b + parents.len(child), (int64_t)u) - b;
    ivec d = dim_by_parent(child);
    if (wh >= parents.len(child) || d.empty()) { err = "child does not list the block as a parent"; return 1; }
    r.push_back(d[wh]); r.push_back(d[wh + 1]);
    return emit(r);
  }
  err = "unknown index name: " + which;
  return 1;
}


// ------------------------------------------------------------------------------------------------ device-resident iteration
// One Gibbs sweep, enqueued only: normals keyed by (seed, row, iteration), Gram refresh and deferred half are the callers'
int Model::enqueue_gibbs(uint64_t seed, bool device_chain, bool draw, bool iloo) {
  if (draw) {  // (draw = false: the previous iteration of the device-resident chain already drew this sweep's normals)
    ST_CUDA(launch_normals(d_z, n_all, seed, device_chain ? 0 : sweep_counter++, d_rowkey, device_chain ? &d_mc->iter : nullptr, stream),
            "normals_kernel");
    n_launches++;
  }
  return gibbs_launch_only(device_chain ? &d_mc->gibbs_fail : d_fail, iloo);
}

// One iteration of spamtree_fit.cpp:167-330 enqueued on the stream without any host synchronisation; every decision is
// taken on the device (st_chain.hpp).  accept_mode: 0 Metropolis rule with a proposal drawn on the device; 1 / 2: the
// proposal is already in the alter slot's theta and is taken / rejected (bench hook).  tev != NULL: CUDA events after the
// phases {start, gibbs, llw, build + accept + deferred half, Gram refresh, tausq + beta}.
int Model::enqueue_iteration(const st_mcmc_opts& o, bool predicting, int accept_mode, bool draws_here, bool draws_next, int record_keep) {
  NvtxRange nvtx("MCMC iteration");
  cudaEvent_t* tev = timing_events_;
  int rc = 0;
  const int nlev = (int)levels.size();
  // Overlap (two streams): theta' and everything of its BUILD that depends on theta alone do not need the new w, so the
  // upper levels of the tree — few work groups each, a chain of latency-bound launches — are built on `stream2` UNDERNEATH
  // the Gibbs sweep and LLW of the main stream, where they cost nothing.  Only the log-density pieces e' prec e need the new
  // w: the levels built early get theirs from an LLW pass over their (few) blocks after the sweep; the big levels are built
  // after the sweep as before (they would only compete with it for the SMs: measured at C4, overlapping everything but the
  // deepest level is slower than no overlap).  Same arithmetic per block as the sequential order.
  const int n_early = n_early_levels_;
  const bool ovl = overlap && o.sample_w && o.sample_theta && n_early >= 1 && stream2 != nullptr;
  bool cond2 = false;  // the accepted-proposal work of this iteration runs on the second stream
  bool prop3 = false;  // the next iteration's proposal runs on the third stream
  if (tev) ST_CUDA(cudaEventRecord(tev[0], stream), "event");
  if (ovl) {
    ST_CUDA(cudaEventRecord(ev_fork, stream), "event");
    ST_CUDA(cudaStreamWaitEvent(stream2, ev_fork, 0), "fork");
    if (tev) ST_CUDA(cudaEventRecord(tev[6], stream2), "event");
    if (accept_mode == 0 && draws_here) { ST_CUDA(launch_mh_propose(d_mc, stream2), "mh_propose_kernel"); n_launches++; }
    rc = launch_build_levels(1, 0, n_early, true, stream2);
    if (rc) return rc;
    if (tev) ST_CUDA(cudaEventRecord(tev[7], stream2), "event");
    ST_CUDA(cudaEventRecord(ev_join, stream2), "event");
  }
  // LLW of the current slot (HBM-bound: it streams every row block once) is not needed before the accept step: on a
  // single-GPU handle it runs on the second stream underneath the BUILD of the proposal (tensor-bound, 10 % of the HBM
  // bandwidth), after the sweep has finished.  (Partitioned handles keep it on the main stream, with their collectives.)
  const bool llw2 = llw_overlap && !part && o.sample_w && o.sample_theta && stream2 != nullptr;
  if (o.sample_w) {  // :183-187
    rc = enqueue_gibbs(o.seed, true, draws_here, record_keep > 0 && (keep_mask & ST_KEEP_LOGLIK_INT));  // (saved iterations only)
    if (rc) return rc;
    if (tev) ST_CUDA(cudaEventRecord(tev[1], stream), "event");
    if (llw2 || ovl) ST_CUDA(cudaEventRecord(ev_sweep, stream), "event");
    if (ovl && o.sample_theta) {
      // log-density pieces of the levels built underneath the sweep: an LLW pass over their blocks with the new w, on the
      // second stream as well — it runs next to the BUILD of the big levels on the main stream and is joined before the
      // reduction.  A childless level that was built forward-half only holds Z instead of G: its pieces come from Z and
      // v = L^-1 w_pa, which the pass over the reference blocks above it leaves in d_vrow row by row.
      ST_CUDA(cudaStreamWaitEvent(stream2, ev_sweep, 0), "fork");
      const bool parked_last = n_early == nlev && levels[nlev - 1].deferrable;
      const int nb_early = (n_early < nlev) ? levels[n_early].slot0 : n_obs_nodes;
      const int nb_plain = parked_last ? levels[nlev - 1].slot0 : nb_early;
      ST_CUDA(launch_llw(dt, dslots, 1, 0, nb_plain, d_w, llw_maxlen_, stream2, parked_last ? d_vrow : nullptr, 0),
              "llw_kernel(early levels of the proposal)");
      n_launches++;
      if (parked_last) {
        ST_CUDA(launch_llw(dt, dslots, 1, nb_plain, nb_early - nb_plain, d_w, llw_maxlen_, stream2, d_vrow, 1), "llw_kernel(parked level)");
        n_launches++;
      }
      ST_CUDA(cudaEventRecord(ev_early_llw, stream2), "event");
    }
    if (llw2) {
      ST_CUDA(cudaStreamWaitEvent(stream2, ev_sweep, 0), "fork");
      if (tev) ST_CUDA(cudaEventRecord(tev[8], stream2), "event");
      ST_CUDA(launch_llw(dt, dslots, 0, 0, n_obs_nodes, d_w, llw_maxlen_, stream2), "llw_kernel");
      n_launches++;
      ST_CUDA(launch_loglik_reduce(dslots, 0, 0, n_obs_nodes, nullptr, d_mc->red_llw, d_red_scratch + kReduceScratch, stream2), "loglik_reduce");
      n_launches++;
      if (tev) ST_CUDA(cudaEventRecord(tev[9], stream2), "event");
      ST_CUDA(cudaEventRecord(ev_llw, stream2), "event");
    } else {
      ST_CUDA(launch_llw(dt, dslots, 0, 0, n_obs_nodes, d_w, llw_maxlen_, stream), "llw_kernel");
      n_launches++;
      rc = reduce_loglik(0, nullptr, d_mc->red_llw, nullptr);
      if (rc) return rc;
    }
  } else if (tev) {
    ST_CUDA(cudaEventRecord(tev[1], stream), "event");
  }
  if (tev) ST_CUDA(cudaEventRecord(tev[2], stream), "event");
  if (o.sample_theta) {  // :203-289
    if (ovl) {
      ST_CUDA(cudaStreamWaitEvent(stream, ev_join, 0), "join");
      rc = launch_build_levels(1, n_early, nlev, false, stream);
      if (rc) return rc;
      ST_CUDA(cudaStreamWaitEvent(stream, ev_early_llw, 0), "join");  // the early levels' log-density pieces (second stream, above)
    } else {
      if (accept_mode == 0 && draws_here) { ST_CUDA(launch_mh_propose(d_mc, stream), "mh_propose_kernel"); n_launches++; }
      rc = launch_build_levels(1, 0, nlev, false, stream);
      if (rc) return rc;
    }
    rc = reduce_loglik(1, d_fail, d_mc->red_build, nullptr);
    if (rc) return rc;
    if (llw2) ST_CUDA(cudaStreamWaitEvent(stream, ev_llw, 0), "join");
    ST_CUDA(launch_mh_accept(d_mc, accept_mode, o.sample_w ? 1 : 0, stream, (int)theta[0].size()), "mh_accept_kernel");
    n_launches++;
    // An accepted proposal: the new param_data's childless level gets its backward half, the message Grams are refreshed.
    // Neither touches w, XB or the chain's scalars: on a single-GPU handle they run on the second stream while the main
    // stream goes on with the prediction, the tausq / beta steps and the tick, and are joined at the end of the iteration
    // (the next sweep needs them).  On the 75 % of the iterations that reject, the ten launches exit at once on their run
    // flag — underneath the same tail instead of in front of it.
    cond2 = !part && stream2 != nullptr;
    cudaStream_t cs = cond2 ? stream2 : stream;
    prop3 = accept_mode == 0 && draws_next && stream3 != nullptr;
    if (cond2 || prop3) ST_CUDA(cudaEventRecord(ev_acc, stream), "event");
    if (cond2) ST_CUDA(cudaStreamWaitEvent(stream2, ev_acc, 0), "fork");
    if (prop3) {
      // the NEXT iteration's proposal needs nothing but this accept step (theta, the adapted proposal covariance): it is drawn
      // now, on a stream of its own underneath the tail, so that the next iteration's BUILD starts without it in front
      ST_CUDA(cudaStreamWaitEvent(stream3, ev_acc, 0), "fork");
      ST_CUDA(launch_mh_propose(d_mc, stream3, 1), "mh_propose_kernel(next iteration)");
      n_launches++;
      ST_CUDA(cudaEventRecord(ev_prop, stream3), "event");
    } else if (accept_mode == 0 && draws_next) {
      ST_CUDA(launch_mh_propose(d_mc, stream, 1), "mh_propose_kernel(next iteration)");
      n_launches++;
    }
    if (tev) ST_CUDA(cudaEventRecord(tev[3], stream), "event");
    if (tev && cond2) ST_CUDA(cudaEventRecord(tev[10], cs), "event");
    rc = launch_deferred_half(0, &d_mc->accepted_now, cs);
    if (rc) return rc;
    if (tev) ST_CUDA(cudaEventRecord(cond2 ? tev[11] : tev[3], cs), "event");
    rc = refresh_grams(&d_mc->accepted_now, cs);
    if (rc) return rc;
    if (tev && cond2) ST_CUDA(cudaEventRecord(tev[12], cs), "event");
    if (cond2) ST_CUDA(cudaEventRecord(ev_cond, stream2), "event");
  } else if (tev) {
    ST_CUDA(cudaEventRecord(tev[3], stream), "event");
  }
  if (tev) ST_CUDA(cudaEventRecord(tev[4], stream), "event");
  if (predicting && o.sample_predicts && o.sample_w && pred_level.nslots > 0) {  // :302-306, predict_std :1234-1358
    ST_CUDA(launch_predict_gate(d_mc, stream), "predict_gate_kernel");
    for (const auto& B : pred_level.build_launches) {
      ST_CUDA(launch_build(2, dt, dslots, 0, d_Hpred, d_sdpred, 0, d_grp_slot0 + B.grp0, d_grp_nn + B.grp0, B.ngrp, d_w, d_fail + 1, B.ns, 0,
                           B.smem, stream, B.threads, nullptr, false, &d_mc->predict_build),
              "build_level_kernel(predict)");
      n_launches++;
    }
    ST_CUDA(launch_predict_sample(dt, pred_level.slot0, pred_level.nslots, d_Hpred, d_sdpred, d_w, d_z, stream), "predict_sample_kernel");
    n_launches += 2;
  }
  if (draws_next && o.sample_w) {
    // the NEXT sweep's normals (Philox counter = iteration + 1), once this iteration's last reader of d_z — the prediction
    // draw — is through: on the third stream, underneath the tail, so that the next sweep starts with its first level
    if (stream3) {
      ST_CUDA(cudaEventRecord(ev_zfree, stream), "event");
      ST_CUDA(cudaStreamWaitEvent(stream3, ev_zfree, 0), "fork");
      ST_CUDA(launch_normals(d_z, n_all, o.seed, 1, d_rowkey, &d_mc->iter, stream3), "normals_kernel(next iteration)");
      ST_CUDA(cudaEventRecord(ev_prop, stream3), "event");
      prop3 = true;
    } else {
      ST_CUDA(launch_normals(d_z, n_all, o.seed, 1, d_rowkey, &d_mc->iter, stream), "normals_kernel(next iteration)");
    }
    n_launches++;
  }
  if (o.sample_tausq || o.sample_beta) {  // :308-330
    rc = enqueue_stats();
    if (rc) return rc;
    ST_CUDA(launch_tausq_beta(d_mc, d_scalars + 8, d_xtx, d_tausq_inv, d_bcoeff, d_bscratch, o.sample_tausq, o.sample_beta, stream, p, q),
            "tausq_beta_kernel");
    n_launches++;
    if (o.sample_beta) { ST_CUDA(launch_xb(dt, n_all, p, d_bcoeff, d_xb, stream), "xb_kernel"); n_launches++; }
  }
  // (the next iteration's proposal reads the iteration counter: it must be through before the tick)
  if (prop3) ST_CUDA(cudaStreamWaitEvent(stream, ev_prop, 0), "join");
  if (record_keep > 0)  // a saved iteration (:376-382): theta, tausq, beta into the device sample arrays, and the tick
    ST_CUDA(launch_record(d_mc, d_tausq_inv, d_bcoeff, d_theta_mcmc, d_beta_mcmc, d_tausq_mcmc, record_keep, stream, 1), "record_kernel");
  else
    ST_CUDA(launch_chain_tick(d_mc, stream), "chain_tick_kernel");
  n_launches++;
  if (tev) ST_CUDA(cudaEventRecord(tev[5], stream), "event");
  if (cond2) ST_CUDA(cudaStreamWaitEvent(stream, ev_cond, 0), "join");
  if (tev) ST_CUDA(cudaEventRecord(tev[13], stream), "event");
  return 0;
}

// brings the host's view of the chain (cur, thetas, log-densities, beta, tausq, the flags of the lazy work) back in step
// with the device after a device-resident run; one synchronisation
int Model::pull_chain_state() {
  ST_CUDA(cudaMemcpyAsync(h_mc, d_mc, sizeof(ChainDev), cudaMemcpyDeviceToHost, stream), "D2H chain");
  ST_CUDA(cudaMemcpyAsync(h_scalars, d_tausq_inv, q * sizeof(double), cudaMemcpyDeviceToHost, stream), "D2H tausq");
  ST_CUDA(cudaMemcpyAsync(h_scalars + 8, d_bcoeff, (size_t)p * q * sizeof(double), cudaMemcpyDeviceToHost, stream), "D2H beta");
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  cur = h_mc->cur;
  for (int sl = 0; sl < 2; sl++) {
    std::copy(h_mc->theta[sl], h_mc->theta[sl] + theta[sl].size(), theta[sl].begin());
    loglik_w[sl] = h_mc->loglik[sl];
    logdetCi[sl] = h_mc->logdet[sl];
  }
  std::copy(h_scalars, h_scalars + q, tausq_inv.begin());
  std::copy(h_scalars + 8, h_scalars + 8 + (size_t)p * q, Bcoeff.begin());
  bool any_def = false;
  for (auto& L : levels) any_def |= L.deferrable;
  deferred_[cur] = false;            // completed on the device whenever a proposal was accepted
  deferred_[1 - cur] = any_def;      // the alter slot holds the forward half of the last proposal
  gram_stale = false;
  pred_H_valid = h_mc->pred_valid != 0;
  stats_valid_mode_ = -1;
  return 0;
}

// state of the device chain before a run / a bench iteration: everything the host-driven path may have changed
int Model::push_chain_state(const st_mcmc_opts* o, uint64_t seed) {
  ChainDev& C = *h_mc;
  const int npar = (int)theta[0].size();
  if (npar > kMaxPar) { err = "more than 64 covariance parameters"; return 4; }
  std::memset(&C, 0, sizeof(ChainDev));
  for (int j = 0; j < q; j++) C.nobs[j] = (double)nobs_by_q[j];
  C.cur = cur; C.npar = npar; C.p = p; C.q = q;
  for (int sl = 0; sl < 2; sl++) {
    std::copy(theta[sl].begin(), theta[sl].end(), C.theta[sl]);
    std::string e2;
    if (!make_covtab(theta[sl].data(), npar, q, C.tab[sl], e2)) { err = e2; return 1; }
    C.loglik[sl] = loglik_w[sl]; C.logdet[sl] = logdetCi[sl];
  }
  std::copy(theta[cur].begin(), theta[cur].end(), C.predict_param);
  C.pred_valid = pred_H_valid ? 1 : 0;
  C.seed = seed;
  if (o) {
    C.adapting = o->adapting;
    std::copy(o->set_unif_bounds, o->set_unif_bounds + 2 * npar, C.bounds);
    if (!ram_init(npar, o->mcmcsd, C.paramsd, C.prodparam)) { err = "mcmcsd is not positive definite"; return 1; }
  }
  // (h_chain is pinned and is not touched again before pull_chain_state's synchronisation: no wait needed here)
  ST_CUDA(cudaMemcpyAsync(d_mc, h_mc, sizeof(ChainDev), cudaMemcpyHostToDevice, stream), "H2D chain");
  // the BUILD failure counter is zero between BUILDs (the reduction that consumes it clears it); make sure it starts so
  ST_CUDA(cudaMemsetAsync(d_fail, 0, 4 * sizeof(int), stream), "memset");
  return 0;
}

// the row-index mode of the beta step on the device (SURVEY App. D #12); one synchronisation when it changes
int Model::set_widx_mode(bool faithful_index) {
  const int mode = faithful_index ? 1 : 0;
  if (beta_widx_mode == mode) return 0;
  const std::vector<int>& src = faithful_index ? beta_widx_faithful : beta_widx_plain;
  ST_CUDA(cudaMemcpyAsync(d_obs_widx, src.data(), n_all * sizeof(int), cudaMemcpyHostToDevice, stream), "H2D widx");
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  beta_widx_mode = mode;
  return 0;
}

// one hot-path iteration with event timing (bench hook): the device-resident iteration with a host-supplied proposal and
// accept decision; the only synchronisation is the one that reads the events and the log-densities back
int Model::bench_iteration(const double* theta_prop, int do_swap, uint64_t seed, double* out3, float* ms_out) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  int rc = complete_slot(cur);
  if (rc) return rc;
  if (gram_stale) { rc = refresh_grams(); if (rc) return rc; }
  rc = set_widx_mode(part ? false : (beta_widx_mode != 0));
  if (rc) return rc;
  rc = push_chain_state(nullptr, seed);  // the device's chain state takes over from the host's
  if (rc) return rc;
  // the proposal into the alter slot (device decides which physical slot that is)
  ThetaPack pk;
  std::string e;
  pk.n = (int)theta[0].size();
  std::copy(theta_prop, theta_prop + pk.n, pk.theta);
  if (!make_covtab(theta_prop, pk.n, q, pk.tab, e)) { err = e; return 1; }
  ST_CUDA(launch_chain_set_theta(d_mc, 1, pk, stream), "chain_set_theta_kernel");
  alter_scratch = false;  // (the iteration builds the alter slot for theta_prop)
  st_mcmc_opts o{};
  o.sample_beta = o.sample_tausq = o.sample_theta = o.sample_w = 1;
  o.seed = seed;
  timing_events_ = ev;
  rc = enqueue_iteration(o, false, do_swap ? 1 : 2, true, false);
  timing_events_ = nullptr;
  if (rc) return rc;
  rc = pull_chain_state();
  if (rc) return rc;
  if (h_mc->gibbs_fail) { err = "Error at gibbs_sample_w: conditional precision not positive definite"; return 3; }
  const bool ok = h_mc->red_build[6] == 0.0;
  out3[0] = loglik_w[1 - cur]; out3[1] = loglik_w[cur]; out3[2] = ok ? 1.0 : 0.0;
  if (h_mc->accepted_now) { out3[0] = loglik_w[cur]; out3[1] = loglik_w[1 - cur]; }  // {proposal, previous current}
  if (ms_out) {
    float t[5], early = 0.f;
    for (int i = 0; i < 5; i++) ST_CUDA(cudaEventElapsedTime(&t[i], ev[i], ev[i + 1]), "elapsed");
    const bool ovl = overlap && n_early_levels_ >= 1 && stream2 != nullptr;
    if (ovl) ST_CUDA(cudaEventElapsedTime(&early, ev[6], ev[7]), "elapsed");
    ms_out[0] = t[0] + t[3];  // GIBBS sweep + the Gram refresh an accepted proposal triggers
    ms_out[1] = t[1];         // LLW
    float dh = 0.f, gr = 0.f;  // single-GPU handles: deferred half and Gram refresh on the second stream, underneath the tail
    if (!part && stream2 != nullptr) {
      ST_CUDA(cudaEventElapsedTime(&dh, ev[10], ev[11]), "elapsed");
      ST_CUDA(cudaEventElapsedTime(&gr, ev[11], ev[12]), "elapsed");
    }
    if (llw_overlap && !part && stream2 != nullptr) ST_CUDA(cudaEventElapsedTime(&ms_out[1], ev[8], ev[9]), "elapsed");  // on the second stream, underneath BUILD
    ms_out[0] += gr;
    ms_out[2] = t[2] + dh;    // BUILD on the main stream + accept + the deferred half of an accepted proposal
    ms_out[3] = t[4];         // tausq + beta
    ST_CUDA(cudaEventElapsedTime(&ms_out[4], ev[0], ev[13]), "elapsed");  // the whole iteration on the main stream
    // the upper levels of BUILD when they run on the second stream, underneath the sweep (elapsed there: it includes the time
    // their thread blocks wait behind the sweep's, so [0..3] + [5] exceeds [4]); 0 when the iteration is sequential
    ms_out[5] = early;
  }
  return 0;
}

// The loop of spamtree_mv_mcmc (spamtree_fit.cpp:167-391) with the chain state in device memory: the host only enqueues
// (one CUDA-graph launch per iteration on a single-GPU handle), saved iterations leave through asynchronous copies, and
// the one synchronisation is at the end of the run.  Random numbers: Philox streams keyed by (seed, row or parameter,
// iteration) — rows by their id in the whole problem, so that a partitioned run draws what a single-GPU run draws.
int Model::chain_run(const st_mcmc_opts& o, st_mcmc_out& out) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  if (part && o.faithful_beta_index) {
    err = "partitioned runs support only the corrected beta row index (faithful_index = 0): the reference's mis-indexing "
          "(SURVEY App. D #12) mixes rows that live on different ranks";
    return 4;
  }
  // the device sample store (st_keep_samples_on_device): sized and checked before anything is allocated or launched, so that a
  // refused run leaves the handle as it was; a run replaces the last run's store
  const bool iloo = (keep_mask & ST_KEEP_LOGLIK_INT) != 0;
  if (iloo && !o.sample_w) {
    err = "st_mcmc_run: the integrated log-likelihood (ST_KEEP_LOGLIK_INT) is formed by the Gibbs sweep over w: it needs sample_w";
    return 1;
  }
  if (keep_mask) {
    if (part) { err = "st_mcmc_run: the device sample store is not supported on partitioned handles"; return 4; }
    const int rc = store.reserve(DrawStore::mask_of(keep_mask), (size_t)n_all * (size_t)std::max(o.keep, 0) * sizeof(double), "st_mcmc_run", err);
    if (rc) return rc;
  }
  double o3[3];
  int rc = get_loglik_comps_w(0, o3);  // spamtree_fit.cpp:110-111
  if (rc) return rc;
  rc = get_loglik_comps_w(1, o3);
  if (rc) return rc;
  rc = complete_slot(cur);
  if (rc) return rc;
  if (gram_stale) { rc = refresh_grams(); if (rc) return rc; }
  rc = set_widx_mode(o.faithful_beta_index != 0);
  if (rc) return rc;
  if (iloo) {
    rc = alloc_loglik_int();
    if (rc) return rc;
    ll_int_valid_ = false;
  }
  const int npar = (int)theta[0].size(), keep = o.keep, mcmc = o.thin * o.keep + o.burn;
  // sample arrays on the device, copied out once at the end
  const size_t n_th = (size_t)npar * keep, n_be = (size_t)p * keep * q, n_ta = (size_t)q * keep;
  if (n_th + n_be + n_ta > samp_cap_ || !d_samp_) {
    if (d_samp_) { cudaFree(d_samp_); d_samp_ = nullptr; }
    samp_cap_ = std::max<size_t>(n_th + n_be + n_ta, 1);
    ST_CUDA(cudaMalloc((void**)&d_samp_, samp_cap_ * sizeof(double)), "alloc samples");
  }
  double* dsamp = d_samp_;
  d_theta_mcmc = dsamp; d_beta_mcmc = dsamp + n_th; d_tausq_mcmc = dsamp + n_th + n_be;
  rc = push_chain_state(&o, o.seed);
  if (rc) return rc;
  // saved rows: w (k = 0) and yhat (k = 1) into the device store and / or the caller's arrays
  double* const host_rows[2] = {out.w_mcmc, out.yhat_mcmc};
  CopyOut co(stream, copy_stream, err);
  if (host_rows[0] || host_rows[1]) {
    rc = co.open({host_rows[0], host_rows[1]}, (size_t)keep * n_all * sizeof(double), 2, n_all);
    if (rc) return rc;
  }
  // one CUDA graph per kind of iteration (with / without prediction); partitioned handles enqueue directly (their
  // collectives are library calls on the stream)
  static const bool no_graph = getenv("ST_GRAPH") && atoi(getenv("ST_GRAPH")) == 0;
  // partitioned handles enqueue every iteration directly.  Capturing the library's NCCL collectives into the graph is
  // possible (ST_PART_GRAPH=1, experimental) and measured: C3 on 2 GPUs 894 against 885 it/s end to end — but one 2-rank run
  // of tools/run_partition.py hung with it, so it is not the default
  static const bool part_graph = getenv("ST_PART_GRAPH") && atoi(getenv("ST_PART_GRAPH")) == 1;
  bool use_graph = !no_graph && (!part || (nccl_comm != nullptr && part_graph));
  // (a graph holds the addresses and the layout of the sample arrays: keep and their base are part of its key; and whether
  // its sweep forms the integrated log-likelihood)
  const long long key_base = ((o.sample_beta ? 1 : 0) | (o.sample_tausq ? 2 : 0) | (o.sample_theta ? 4 : 0) | (o.sample_w ? 8 : 0) | (o.sample_predicts ? 16 : 0) |
                              (iloo ? 32 : 0)) +
                             64LL * keep + (long long)(reinterpret_cast<uintptr_t>(d_samp_) >> 4) * 1000003LL;
  int msaved = 0;
  const auto t0 = std::chrono::steady_clock::now();
  for (int m = 0; m < mcmc; m++) {
    const int mx = m - o.burn;
    const bool saved = mx >= 0 && mx % o.thin == 0;
    const bool predicting = saved;
    const int which = predicting ? 1 : 0;
    bool launched = false;
    // The proposal of iteration m + 1 is drawn inside iteration m, right after its accept step; iteration 0 draws its own as
    // well and the last one draws none (the alter slot's theta then stays the proposal that was built).  Both run directly.
    const bool first = m == 0, last = m + 1 == mcmc;
    if (use_graph && !first && !last) {  // (iteration 0 runs directly: it also sets the kernels' shared-memory attributes)
      if (graph_key_[which] != key_base || !graph_exec_[which]) {
        if (graph_exec_[which]) { cudaGraphExecDestroy((cudaGraphExec_t)graph_exec_[which]); graph_exec_[which] = nullptr; }
        cudaGraph_t g = nullptr;
        const double nl0 = n_launches;
        bool ok = cudaStreamBeginCapture(stream, cudaStreamCaptureModeRelaxed) == cudaSuccess;
        int rcc = ok ? enqueue_iteration(o, predicting, 0, false, true, saved ? keep : 0) : 0;
        if (ok) ok = (cudaStreamEndCapture(stream, &g) == cudaSuccess) && g && rcc == 0;
        cudaGraphExec_t ge = nullptr;
        if (ok) ok = cudaGraphInstantiate(&ge, g, 0) == cudaSuccess;
        if (g) cudaGraphDestroy(g);
        if (ok) { graph_exec_[which] = ge; graph_key_[which] = key_base; graph_launches_[which] = n_launches - nl0; }
        else { (void)cudaGetLastError(); use_graph = false; }
        n_launches = nl0;  // (capturing enqueues nothing)
      }
      if (use_graph) {
        ST_CUDA(cudaGraphLaunch((cudaGraphExec_t)graph_exec_[which], stream), "cudaGraphLaunch");
        n_launches += graph_launches_[which];
        launched = true;
      }
    }
    if (!launched) { rc = enqueue_iteration(o, predicting, 0, first, !last, saved ? keep : 0); if (rc) return rc; }
    if (saved) {  // :376-389
      const size_t off = (size_t)msaved * n_all;
      for (int k = 0; k < 2; k++) {
        const bool kept = (keep_mask & (1 << k)) != 0;
        if (!host_rows[k] && !kept) continue;
        rc = save_rows(co, k, kept ? store.get(k).d + off : nullptr, host_rows[k] ? host_rows[k] + off : nullptr);
        if (rc) return rc;
      }
      if (iloo) {  // this iteration's sweep formed it: into its slot of the store, in boundary order
        ST_CUDA(launch_permute(d_ll_int_, store.get(DrawStore::kLoglikInt).d + off, d_iperm, n_all, stream), "permute_kernel");
        n_launches++;
      }
      msaved++;
    }
  }
  // the one synchronisation of the run: chain state, samples, the saves in flight
  rc = pull_chain_state();
  if (rc) return rc;
  rc = co.finish();
  if (rc) return rc;
  dvec hs(std::max<size_t>(n_th + n_be + n_ta, 1));
  ST_CUDA(cudaMemcpy(hs.data(), dsamp, (n_th + n_be + n_ta) * sizeof(double), cudaMemcpyDeviceToHost), "D2H samples");
  out.mcmc_time = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  if (out.theta_mcmc) std::copy(hs.begin(), hs.begin() + n_th, out.theta_mcmc);
  if (out.beta_mcmc) std::copy(hs.begin() + n_th, hs.begin() + n_th + n_be, out.beta_mcmc);
  if (out.tausq_mcmc) std::copy(hs.begin() + n_th + n_be, hs.end(), out.tausq_mcmc);
  if (out.paramsd) std::copy(h_mc->paramsd, h_mc->paramsd + (size_t)npar * npar, out.paramsd);
  out.n_accepted = h_mc->n_accepted;
  out.n_chol_fail = h_mc->n_chol_fail;
  if (h_mc->gibbs_fail) { err = "Error at gibbs_sample_w: conditional precision not positive definite"; return 3; }
  if (h_mc->nan_loglik) { err = "At nan loglik: error."; return 5; }
  if (iloo && keep > 0) ll_int_valid_ = true;
  if (keep_mask && keep > 0) {  // the run completed: its store and the samples st_predict_new_stored predicts from
    store.commit(DrawStore::mask_of(keep_mask), n_all, keep);
    store.samples.assign(hs.begin(), hs.begin() + (n_th + n_be + n_ta));
  }
  return 0;
}

// ---- the device draw store
int DrawStore::reserve(int mask, size_t bytes_each, const char* what, std::string& err) {
  const int group = ((mask & kRun) ? kRun : 0) | ((mask & kPrediction) ? kPrediction : 0);
  size_t need = 0, reusable = 0;
  for (int k = 0; k < kStores; k++) {
    if (mask & (1 << k)) need += bytes_each;
    if (group & (1 << k)) reusable += s_[k].cap;
  }
  size_t fr = 0, tot = 0;
  if (const cudaError_t e = cudaMemGetInfo(&fr, &tot)) { err = std::string("CUDA error in cudaMemGetInfo: ") + cudaGetErrorString(e); return 2; }
  if (need > fr + reusable) {
    err = std::string(what) + ": the device sample store needs " + std::to_string(need) + " bytes and " + std::to_string(fr + reusable) +
          " bytes of device memory are free";
    return 4;
  }
  if (group & kRun) samples.clear();
  const size_t bytes = std::max<size_t>(bytes_each, 8);
  for (int k = 0; k < kStores; k++) {
    if (!(group & (1 << k))) continue;
    Store& s = s_[k];
    s.S = 0;
    if (!(mask & (1 << k))) { if (s.d) cudaFree(s.d); s = Store(); continue; }
    if (bytes <= s.cap) continue;
    if (s.d) cudaFree(s.d);
    s = Store();
    if (cudaMalloc((void**)&s.d, bytes) != cudaSuccess) {
      (void)cudaGetLastError();
      s.d = nullptr;
      err = std::string(what) + ": allocating " + std::to_string(bytes_each) + " bytes for the device sample store failed";
      return 4;
    }
    s.cap = bytes;
  }
  return 0;
}

void DrawStore::commit(int mask, int64_t n, int S) {
  for (int k = 0; k < kStores; k++)
    if (mask & (1 << k)) { s_[k].n = n; s_[k].S = S; }
}

const DrawStore::Store* DrawStore::find(int which, const std::string& who, std::string& err) const {
  static const char* names[kStores] = {"w", "yhat", "w_new", "y_new", "the integrated log-likelihood"};
  const Store& s = s_[which];
  if (s.d && s.S >= 1) return &s;
  err = who + "no stored draws of " + names[which] +
        (which == kLoglikInt ? " (st_keep_samples_on_device with ST_KEEP_LOGLIK_INT before a device-resident st_mcmc_run that samples w)"
         : which < 2         ? " (st_keep_samples_on_device before a device-resident st_mcmc_run)"
                             : " (st_predict_new_stored with keep_draws)");
  return nullptr;
}

void DrawStore::release() {
  for (Store& s : s_) {
    if (s.d) cudaFree(s.d);
    s = Store();
  }
  samples.clear();
}

int Model::keep_samples_on_device(int what) {
  if (what < 0 || what > (ST_KEEP_W | ST_KEEP_YHAT | ST_KEEP_LOGLIK_INT)) {
    err = "st_keep_samples_on_device: what must be a mask of ST_KEEP_W | ST_KEEP_YHAT | ST_KEEP_LOGLIK_INT";
    return 1;
  }
  if (what && !stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  if (what && part) { err = "st_keep_samples_on_device: partitioned handles are not supported"; return 4; }
  keep_mask = what;
  if (what == 0) {
    if (stream) cudaStreamSynchronize(stream);
    store.release();
  }
  return 0;
}

int Model::summarize(int which, const double* probs, int n_probs, st_summary_out& out) {
  if (which < 0 || which > 3) { err = "st_summarize: which must be 0 (w), 1 (yhat), 2 (w_new) or 3 (y_new)"; return 1; }
  out.n_rows = 0;
  out.n_samples = 0;
  const DrawStore::Store* sp = store.find(which, "st_summarize: ", err);
  if (!sp) return 1;
  const DrawStore::Store& s = *sp;
  if (const int rc = probs_check("st_summarize", probs, n_probs, err)) return rc;
  const size_t cap = 227 * 1024;
  const int R = summary_rows_per_cta(s.S, cap);
  if (R < 1) {
    err = "st_summarize: " + std::to_string(s.S) + " draws per row exceed what one CTA stages in shared memory (at most " +
          std::to_string((cap - (size_t)kSummaryThreads * sizeof(double)) / sizeof(unsigned long long)) + ")";
    return 4;
  }
  out.n_rows = s.n;
  out.n_samples = s.S;
  double* hdst[5] = {out.mean, out.sd, out.quantiles, out.mcse, out.ess};
  if (!(hdst[0] || hdst[1] || hdst[2] || hdst[3] || hdst[4]) || s.n == 0) return 0;
  // one device buffer: mean | sd | mcse | ess | quantiles (n x n_probs) | probs
  const size_t n = (size_t)s.n, nd = (4 + (size_t)n_probs) * n + (size_t)n_probs;
  double* d = nullptr;
  ST_CUDA(cudaMalloc((void**)&d, nd * sizeof(double)), "alloc summaries");
  struct Free { double* p; ~Free() { cudaFree(p); } } fr{d};
  struct StreamSync { cudaStream_t s; ~StreamSync() { cudaStreamSynchronize(s); } } ssync{stream};
  double* dq = d + 4 * n;
  double* dp = dq + (size_t)n_probs * n;
  if (n_probs) ST_CUDA(cudaMemcpyAsync(dp, probs, n_probs * sizeof(double), cudaMemcpyHostToDevice, stream), "H2D probs");
  ST_CUDA(launch_summary(s.d, s.n, s.S, R, dp, n_probs, d, d + n, dq, d + 2 * n, d + 3 * n, stream), "summary_kernel");
  n_launches++;
  const double* dsrc[5] = {d, d + n, dq, d + 2 * n, d + 3 * n};
  for (int c = 0; c < 5; c++) {
    const size_t cnt = c == 2 ? (size_t)n_probs * n : n;
    if (hdst[c] && cnt) ST_CUDA(cudaMemcpyAsync(hdst[c], dsrc[c], cnt * sizeof(double), cudaMemcpyDeviceToHost, stream), "D2H summaries");
  }
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  return 0;
}

int Model::copy_store(int which, double* out, int64_t* n_rows, int32_t* n_samples) {
  if (which < 0 || which >= DrawStore::kStores) {
    err = "st_copy_store: which must be 0 (w), 1 (yhat), 2 (w_new), 3 (y_new) or 4 (the integrated log-likelihood)";
    return 1;
  }
  const DrawStore::Store* sp = store.find(which, "st_copy_store: ", err);
  if (!sp) return 1;
  if (n_rows) *n_rows = sp->n;
  if (n_samples) *n_samples = sp->S;
  if (!out || sp->n == 0) return 0;
  ST_CUDA(cudaStreamSynchronize(stream), "sync");  // (the run or prediction that wrote it)
  ST_CUDA(cudaMemcpy(out, sp->d, (size_t)sp->n * sp->S * sizeof(double), cudaMemcpyDeviceToHost), "D2H store");
  return 0;
}

// ---- several chains (st_summarize_chains, st_summarize_draws; DESIGN.md §5d)
static const size_t kChainsSmemCap = 227 * 1024;

int probs_check(const char* what, const double* probs, int n_probs, std::string& err) {
  if (n_probs < 0 || (n_probs > 0 && !probs)) { err = std::string(what) + ": n_probs < 0, or probs missing"; return 1; }
  for (int j = 0; j < n_probs; j++)
    if (!(probs[j] >= 0.0 && probs[j] <= 1.0)) { err = std::string(what) + ": every prob must lie in [0, 1] (NaN is refused)"; return 1; }
  return 0;
}

int chains_check(const char* what, int K, int S, const double* probs, int n_probs, std::string& err) {
  if (K < 1 || S < 1) { err = std::string(what) + ": n_chains and n_samples must be at least 1"; return 1; }
  if (const int rc = probs_check(what, probs, n_probs, err)) return rc;
  if (chains_rows_per_cta(K, S, kChainsSmemCap) < 1) {
    err = std::string(what) + ": " + std::to_string(K) + " chains of " + std::to_string(S) + " draws exceed what one CTA stages in "
          "shared memory (n_chains x (n_samples + 1) = " + std::to_string((long long)K * (S + 1)) + ", at most " +
          std::to_string((kChainsSmemCap - (size_t)kSummaryThreads * sizeof(double)) / (2 * sizeof(double))) + ")";
    return 4;
  }
  return 0;
}

int summarize_chains(const double* const* src, int64_t n, int K, int S, const double* probs, int n_probs, st_chains_summary_out& out,
                     cudaStream_t st, std::string& err) {
  out.n_rows = n;
  out.n_chains = K;
  out.n_samples = S;
  double* hdst[6] = {out.mean, out.sd, out.quantiles, out.rhat, out.ess_bulk, out.ess_tail};
  if (!(hdst[0] || hdst[1] || hdst[2] || hdst[3] || hdst[4] || hdst[5]) || n == 0) return 0;
  // one device buffer: mean | sd | rhat | ess_bulk | ess_tail | quantiles (n x n_probs) | probs | the K chain pointers
  const size_t nn = (size_t)n, nd = (5 + (size_t)n_probs) * nn + (size_t)n_probs + (size_t)K;
  double* d = nullptr;
  cudaError_t e = cudaMalloc((void**)&d, nd * sizeof(double));
  if (e != cudaSuccess) { (void)cudaGetLastError(); err = std::string("CUDA error in alloc summaries: ") + cudaGetErrorString(e); return 2; }
  struct Free { double* p; ~Free() { cudaFree(p); } } fr{d};
  double* dq = d + 5 * nn;
  double* dp = dq + (size_t)n_probs * nn;
  const double** dsrc = reinterpret_cast<const double**>(dp + n_probs);
  const double* outs[6] = {d, d + nn, dq, d + 2 * nn, d + 3 * nn, d + 4 * nn};
  auto chk = [&](cudaError_t c, const char* what) {
    if (c != cudaSuccess && e == cudaSuccess) { e = c; err = std::string("CUDA error in ") + what + ": " + cudaGetErrorString(c); }
  };
  if (n_probs) chk(cudaMemcpyAsync(dp, probs, n_probs * sizeof(double), cudaMemcpyHostToDevice, st), "H2D probs");
  chk(cudaMemcpyAsync(dsrc, src, K * sizeof(double*), cudaMemcpyHostToDevice, st), "H2D chain pointers");
  if (e == cudaSuccess)
    chk(launch_chains_summary(dsrc, n, K, S, chains_rows_per_cta(K, S, kChainsSmemCap), dp, n_probs, d, d + nn, dq, d + 2 * nn,
                              d + 3 * nn, d + 4 * nn, st),
        "chains_summary_kernel");
  for (int c = 0; c < 6 && e == cudaSuccess; c++) {
    const size_t cnt = c == 2 ? (size_t)n_probs * nn : nn;
    if (hdst[c] && cnt) chk(cudaMemcpyAsync(hdst[c], outs[c], cnt * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H summaries");
  }
  chk(cudaStreamSynchronize(st), "sync");  // (before the buffer is freed, whatever failed)
  return e == cudaSuccess ? 0 : 2;
}

// ---- model criteria (st_fit_criteria, st_fit_criteria_loglik; DESIGN.md §5e)
int criteria_check(const char* what, int K, int S, double r_eff, std::string& err) {
  if (K < 1 || S < 1) { err = std::string(what) + ": n_chains and n_samples must be at least 1"; return 1; }
  if (!(r_eff > 0.0) || !std::isfinite(r_eff)) { err = std::string(what) + ": r_eff must be positive and finite"; return 1; }
  const size_t lim = (kChainsSmemCap - (size_t)kSummaryThreads * sizeof(double)) / sizeof(unsigned long long);
  if ((long long)K * S > (long long)lim || summary_rows_per_cta(K * S, kChainsSmemCap) < 1) {
    err = std::string(what) + ": " + std::to_string(K) + " chains of " + std::to_string(S) + " draws exceed what one CTA stages in "
          "shared memory (n_chains x n_samples = " + std::to_string((long long)K * S) + ", at most " + std::to_string(lim) + ")";
    return 4;
  }
  return 0;
}

int fit_criteria(const double* const* src, int64_t n, int K, int S, double r_eff, const std::vector<char>& obs, const CritInputs* in,
                 st_fit_criteria_out& out, cudaStream_t st, std::string& err) {
  const double nan = std::numeric_limits<double>::quiet_NaN();
  const int N = K * S;
  out.n_rows = n;
  out.n_chains = K;
  out.n_samples = S;
  out.n_obs = 0;
  for (int64_t i = 0; i < n; i++) out.n_obs += obs[i] != 0;
  out.k_threshold = std::min(1.0 - 1.0 / std::log10((double)N), 0.7);
  out.n_k_high = out.n_p_waic_high = 0;
  double* tot[16] = {&out.elpd_loo_total, &out.se_elpd_loo, &out.p_loo_total, &out.looic, &out.se_looic, &out.elpd_waic_total,
                     &out.se_elpd_waic, &out.p_waic_total, &out.waic, &out.se_waic, &out.lpd_total, &out.dbar, &out.dhat,
                     &out.p_dic, &out.dic, nullptr};
  for (int c = 0; tot[c]; c++) *tot[c] = nan;
  double* hdst[6] = {out.lpd, out.elpd_loo, out.p_loo, out.pareto_k, out.elpd_waic, out.p_waic};
  if (!(hdst[0] || hdst[1] || hdst[2] || hdst[3] || hdst[4] || hdst[5]) || n == 0) return 0;
  // one device buffer: the 8 per-row outputs | K chain pointers | with parameters: y | X | bbar | tbar | beta | tausq | mvq
  const size_t nn = (size_t)n, p = in ? in->p : 0, q = in ? in->q : 0;
  const size_t n_par = in ? nn + nn * p + p * q + q + (size_t)N * p * q + (size_t)N * q + (nn + 1) / 2 : 0;
  const size_t nd = 8 * nn + (size_t)K + n_par;
  double* d = nullptr;
  cudaError_t e = cudaMalloc((void**)&d, nd * sizeof(double));
  if (e != cudaSuccess) { (void)cudaGetLastError(); err = std::string("CUDA error in alloc criteria: ") + cudaGetErrorString(e); return 2; }
  struct Free { double* p; ~Free() { cudaFree(p); } } fr{d};
  auto chk = [&](cudaError_t c, const char* what) {
    if (c != cudaSuccess && e == cudaSuccess) { e = c; err = std::string("CUDA error in ") + what + ": " + cudaGetErrorString(c); }
  };
  const double** dsrc = reinterpret_cast<const double**>(d + 8 * nn);
  chk(cudaMemcpyAsync(dsrc, src, K * sizeof(double*), cudaMemcpyHostToDevice, st), "H2D chain pointers");
  CritParams P{};
  dvec bbar, tbar;
  std::vector<int> mvq;
  if (in) {  // (host vectors the copies read stay alive until the synchronisation at the end)
    bbar.assign(p * q, 0.0);
    tbar.assign(q, 0.0);
    for (int g = 0; g < N; g++) {  // pooled means over the N draws, in draw order
      for (size_t c = 0; c < p * q; c++) bbar[c] += in->beta[(size_t)g * p * q + c];
      for (size_t j = 0; j < q; j++) tbar[j] += in->tausq[(size_t)g * q + j];
    }
    for (double& v : bbar) v /= N;
    for (double& v : tbar) v /= N;
    mvq.resize(nn);
    for (size_t i = 0; i < nn; i++) mvq[i] = (int)in->mv_id[i] - 1;
    double* a = d + 8 * nn + K;
    double* dy = a; a += nn;
    double* dX = a; a += nn * p;
    double* dbb = a; a += p * q;
    double* dtb = a; a += q;
    double* dbe = a; a += (size_t)N * p * q;
    double* dta = a; a += (size_t)N * q;
    int* dmv = reinterpret_cast<int*>(a);
    chk(cudaMemcpyAsync(dy, in->y, nn * sizeof(double), cudaMemcpyHostToDevice, st), "H2D y");
    if (p) chk(cudaMemcpyAsync(dX, in->X, nn * p * sizeof(double), cudaMemcpyHostToDevice, st), "H2D X");
    if (p) chk(cudaMemcpyAsync(dbb, bbar.data(), p * q * sizeof(double), cudaMemcpyHostToDevice, st), "H2D beta means");
    chk(cudaMemcpyAsync(dtb, tbar.data(), q * sizeof(double), cudaMemcpyHostToDevice, st), "H2D tausq means");
    if (p) chk(cudaMemcpyAsync(dbe, in->beta, (size_t)N * p * q * sizeof(double), cudaMemcpyHostToDevice, st), "H2D beta samples");
    chk(cudaMemcpyAsync(dta, in->tausq, (size_t)N * q * sizeof(double), cudaMemcpyHostToDevice, st), "H2D tausq samples");
    chk(cudaMemcpyAsync(dmv, mvq.data(), nn * sizeof(int), cudaMemcpyHostToDevice, st), "H2D mv_id");
    P = CritParams{dy, dX, dmv, dbe, dta, dbb, dtb, (int)p, (int)q};
  }
  if (e == cudaSuccess)
    chk(launch_fit_criteria(dsrc, n, K, S, summary_rows_per_cta(N, kChainsSmemCap), r_eff, P, d, st), "fit_criteria_kernel");
  dvec h(8 * nn);
  if (e == cudaSuccess) chk(cudaMemcpyAsync(h.data(), d, 8 * nn * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H criteria");
  chk(cudaStreamSynchronize(st), "sync");  // (before the buffer is freed, whatever failed)
  if (e != cudaSuccess) return 2;
  for (int c = 0; c < 6; c++)
    if (hdst[c]) std::copy(h.begin() + c * nn, h.begin() + (c + 1) * nn, hdst[c]);
  // ---- totals over the observed rows, in row order
  const double* lpd = h.data();
  const double *el = lpd + nn, *pl = el + nn, *kh = pl + nn, *ew = kh + nn, *pw = ew + nn, *db = pw + nn, *dh = db + nn;
  double s[7] = {0, 0, 0, 0, 0, 0, 0};  // elpd_loo, p_loo, elpd_waic, p_waic, lpd, dbar, dhat
  for (size_t i = 0; i < nn; i++) {
    if (!obs[i]) continue;
    s[0] += el[i]; s[1] += pl[i]; s[2] += ew[i]; s[3] += pw[i]; s[4] += lpd[i]; s[5] += db[i]; s[6] += dh[i];
    out.n_k_high += kh[i] > out.k_threshold;
    out.n_p_waic_high += pw[i] > 0.4;
  }
  const double no = (double)out.n_obs;
  auto se = [&](const double* v, double total) {  // sqrt(n_obs var(v_i, ddof 1))
    const double m = total / no;
    double ss = 0.0;
    for (size_t i = 0; i < nn; i++)
      if (obs[i]) ss += (v[i] - m) * (v[i] - m);
    return out.n_obs > 1 ? std::sqrt(no * ss / (no - 1)) : nan;
  };
  out.elpd_loo_total = s[0];
  out.se_elpd_loo = se(el, s[0]);
  out.p_loo_total = s[1];
  out.looic = -2.0 * s[0];
  out.se_looic = 2.0 * out.se_elpd_loo;
  out.elpd_waic_total = s[2];
  out.se_elpd_waic = se(ew, s[2]);
  out.p_waic_total = s[3];
  out.waic = -2.0 * s[2];
  out.se_waic = 2.0 * out.se_elpd_waic;
  out.lpd_total = s[4];
  if (in) {
    out.dbar = s[5];
    out.dhat = s[6];
    out.p_dic = s[5] - s[6];
    out.dic = s[5] + out.p_dic;
  }
  return 0;
}


// ------------------------------------------------------------------------------------------------------ predict_new
// Posterior predictive draws at new rows from saved samples (DESIGN.md, "Prediction at new locations").  The new rows are
// laid out as extra nodes behind the tree: rows of one parent chain, split into pseudo-blocks narrow enough for one BUILD
// work group (they are conditionally independent, so any split is exact), appended to temporary copies of the per-node and
// per-row arrays.  Per sample: BUILD of the reference levels into the alter slot when theta changed, w_s into node order,
// build_level_kernel<3> (forward sweep only: mean and sd per row), predict_draw_kernel; the draws leave on a copy stream.
// from_store: the samples are the last stored run's (theta / beta / tausq from its host copy, w_s gathered straight from the
// device store); keep_draws: w_new / y_new are written into the prediction's device store instead of scratch.
int Model::predict_new(const st_new_rows& R, const st_pred_samples& PS_in, st_pred_out& out, bool from_store, bool keep_draws) {
  if (!stream) { err = "this handle has no device state (created with device < 0)"; return 2; }
  if (part) { err = "predict_new: partitioned handles are not supported"; return 4; }
  out.n_builds = 0;
  const int npar = (int)theta[0].size();
  st_pred_samples PS = PS_in;
  if (from_store) {  // (a stored w comes with the run's samples: DrawStore::commit)
    const DrawStore::Store* sw = store.find(0, "st_predict_new_stored: ", err);
    if (!sw) return 1;
    const int Ss = sw->S;
    PS.n_samples = Ss;
    PS.theta = store.samples.data();
    PS.beta = PS.theta + (size_t)npar * Ss;
    PS.tausq = PS.beta + (size_t)p * Ss * q;
    PS.w = sw->d;  // (a device pointer: read by gather_sample_kernel only)
    PS.w_row_stride = 1;
    PS.w_sample_stride = n_all;
    PS.z = PS.eps = nullptr;
  }
  const int64_t nn = R.n_new;
  const int S = PS.n_samples;
  if (nn < 0 || S < 0) { err = "predict_new: negative n_new or n_samples"; return 1; }
  if (keep_draws) {  // checked before anything is allocated; the previous prediction's store is replaced
    const int rc = store.reserve(DrawStore::kPrediction, (size_t)std::max<int64_t>(nn, 0) * S * sizeof(double), "st_predict_new_stored", err);
    if (rc) return rc;
  }
  if (nn == 0 || S == 0) return 0;
  if (!R.coords || !R.mv_id || !R.group || !R.parents_ptr || R.n_groups < 1 || !PS.theta || !PS.beta || !PS.tausq || !PS.w) {
    err = "predict_new: a required input is missing";
    return 1;
  }
  if (nn >= (1LL << 31) - n_all) { err = "predict_new: too many new rows"; return 4; }
  const int64_t ng = R.n_groups;
  if (R.parents_ptr[0] != 0) { err = "predict_new: parents_ptr[0] must be 0"; return 1; }
  for (int64_t g = 0; g < ng; g++)
    if (R.parents_ptr[g + 1] <= R.parents_ptr[g]) { err = "predict_new: a group has no parents (or parents_ptr decreases)"; return 1; }
  if (!R.parents_idx) { err = "predict_new: parents_idx missing"; return 1; }
  // every group's parents must be a chain of observed reference blocks: parents(lp) followed by lp (limited: lp alone)
  std::vector<int> glast(ng);
  for (int64_t g = 0; g < ng; g++) {
    const int64_t* pl = R.parents_idx + R.parents_ptr[g];
    const int64_t np = R.parents_ptr[g + 1] - R.parents_ptr[g];
    for (int64_t t = 0; t < np; t++)
      if (pl[t] < 0 || pl[t] >= n_blocks) { err = "predict_new: a parent id is outside 0..n_blocks-1"; return 1; }
    const int64_t lp = pl[np - 1];
    const int sl = slot_of_block[lp];
    if (sl < 0 || sl >= n_obs_nodes || block_ct_obs[lp] == 0 || !block_is_reference[lp]) {
      err = "predict_new: the last parent of a group is not an observed reference block";
      return 1;
    }
    if (limited ? np != 1 : (parents.len(lp) != np - 1 || !std::equal(parents.row(lp), parents.row(lp) + (np - 1), pl))) {
      err = limited ? "predict_new: limited_tree = TRUE: a group lists more than one parent"
                    : "predict_new: a group's parents are not the ancestor chain of its last parent";
      return 1;
    }
    glast[g] = sl;
  }
  for (int64_t i = 0; i < nn; i++) {
    if (R.group[i] < 0 || R.group[i] >= ng) { err = "predict_new: a group id is outside 0..n_groups-1"; return 1; }
    if (R.mv_id[i] < 1 || R.mv_id[i] > q) { err = "predict_new: mv_id outside 1..q"; return 1; }
    if (!std::isfinite(R.coords[i]) || !std::isfinite(R.coords[i + nn])) { err = "predict_new: coords hold a non-finite value"; return 1; }
  }
  const bool cmaj = PS.w_row_stride == 1 && PS.w_sample_stride >= n_all;  // one sample per contiguous column
  const bool rmaj = PS.w_sample_stride == 1 && PS.w_row_stride >= S;       // one row's samples contiguous
  if (!cmaj && !rmaj) { err = "predict_new: w strides must be (1, >= n_all) or (>= n_samples, 1)"; return 1; }
  for (int s = 0; s < S; s++)
    for (int j = 0; j < q; j++)
      if (!(PS.tausq[j + (size_t)s * q] >= 0.0)) { err = "predict_new: tausq must be non-negative"; return 1; }

  // ---- layout: rows by parent chain (slot of the last parent), caller order inside; pseudo-blocks of at most mcap rows
  std::vector<int64_t> lay2row(nn);
  std::iota(lay2row.begin(), lay2row.end(), 0);
  std::stable_sort(lay2row.begin(), lay2row.end(), [&](int64_t a, int64_t b) { return glast[R.group[a]] < glast[R.group[b]]; });
  const int wmax = kBuildMaxThreads / 32;
  const int col_cap = std::min(max_group_cols, kMaxGroupCols);
  std::vector<int> pm, prow0, pk, pP, pchoff, pchain, pcpoff;
  std::vector<long long> prioff;
  for (int64_t k0 = 0; k0 < nn;) {
    const int lp = glast[R.group[lay2row[k0]]];
    int64_t k1 = k0;
    while (k1 < nn && glast[R.group[lay2row[k1]]] == lp) k1++;
    // the chain: the parent's own chain + the parent (limited trees: the parent alone, its marginal factor)
    std::vector<int> ch;
    if (!limited) ch.assign(h_chain.begin() + h_chain_off[lp], h_chain.begin() + h_chain_off[lp] + h_k[lp]);
    ch.push_back(lp);
    if ((int)ch.size() > kMaxChain) { err = "predict_new: ancestor chains longer than 32 are not supported"; return 4; }
    int P = 0;
    std::vector<int> poff;
    for (int a : ch) { poff.push_back(P); P += h_m[a]; }
    int mcap = col_cap - 1;  // (the w_pa column takes one)
    while (mcap >= 1 && build_plan(P, mcap + 1, 0, mcap, 1, 0, wmax).total > smem_budget) mcap--;
    if (mcap < 1) { err = "predict_new: a parent set is too large for one BUILD work group (P=" + std::to_string(P) + ")"; return 4; }
    for (int64_t b0 = k0; b0 < k1; b0 += mcap) {
      const int m = (int)std::min<int64_t>(mcap, k1 - b0);
      pm.push_back(m); prow0.push_back((int)(n_all + b0)); prioff.push_back(b0);
      pk.push_back((int)ch.size()); pP.push_back(P); pchoff.push_back((int)(h_chain.size() + pchain.size()));
      pchain.insert(pchain.end(), ch.begin(), ch.end());
      pcpoff.insert(pcpoff.end(), poff.begin(), poff.end());
    }
    k0 = k1;
  }
  const int npb = (int)pm.size();
  // work groups: one pseudo-block each (pseudo-blocks of one chain are already as wide as a group may be), bucketed by
  // width as make_groups buckets a level's groups
  std::vector<GroupSpec> specs;
  for (int t = 0; t < npb; t++) specs.push_back({n_nodes + t, 1, build_plan(pP[t], pm[t] + 1, 0, pm[t], 1, 0, wmax).NT});
  std::vector<LevelInfo::BuildLaunch> launches;
  std::vector<int> gslot0, gnn;
  bucket_groups(specs, [&](const GroupSpec& g, int ns, int nw) {
    const int t = g.s - n_nodes;
    return build_plan(pP[t], pm[t] + 1, 0, pm[t], ns, 0, nw).total;
  }, gslot0, gnn, launches);

  // ---- temporary device state (freed on every exit)
  struct Scratch {
    std::vector<void*> dev;
    ~Scratch() { for (void* p : dev) cudaFree(p); }
  } X;
  auto dalloc = [&](void** p, size_t bytes) -> cudaError_t {
    cudaError_t e = cudaMalloc(p, std::max<size_t>(bytes, 8));
    if (e == cudaSuccess) X.dev.push_back(*p);
    return e;
  };
  // make sure the stream is idle before the scratch is freed on an early exit
  struct StreamSync { cudaStream_t s; ~StreamSync() { cudaStreamSynchronize(s); } } ssync{stream};
  const int64_t nrow2 = n_all + nn;
  double *d_cx2, *d_cy2;
  int* d_mvq2;
  ST_CUDA(dalloc((void**)&d_cx2, nrow2 * sizeof(double)), "alloc");
  ST_CUDA(dalloc((void**)&d_cy2, nrow2 * sizeof(double)), "alloc");
  ST_CUDA(dalloc((void**)&d_mvq2, nrow2 * sizeof(int)), "alloc");
  ST_CUDA(cudaMemcpyAsync(d_cx2, dt.cx, n_all * sizeof(double), cudaMemcpyDeviceToDevice, stream), "D2D cx");
  ST_CUDA(cudaMemcpyAsync(d_cy2, dt.cy, n_all * sizeof(double), cudaMemcpyDeviceToDevice, stream), "D2D cy");
  ST_CUDA(cudaMemcpyAsync(d_mvq2, dt.mvq, n_all * sizeof(int), cudaMemcpyDeviceToDevice, stream), "D2D mvq");
  dvec ncx(nn), ncy(nn);
  std::vector<int> nmvq(nn), cmvq(nn);
  for (int64_t k = 0; k < nn; k++) {
    const int64_t i = lay2row[k];
    ncx[k] = R.coords[i]; ncy[k] = R.coords[i + nn]; nmvq[k] = (int)R.mv_id[i] - 1;
  }
  for (int64_t i = 0; i < nn; i++) cmvq[i] = (int)R.mv_id[i] - 1;
  ST_CUDA(cudaMemcpyAsync(d_cx2 + n_all, ncx.data(), nn * sizeof(double), cudaMemcpyHostToDevice, stream), "H2D new rows");
  ST_CUDA(cudaMemcpyAsync(d_cy2 + n_all, ncy.data(), nn * sizeof(double), cudaMemcpyHostToDevice, stream), "H2D new rows");
  ST_CUDA(cudaMemcpyAsync(d_mvq2 + n_all, nmvq.data(), nn * sizeof(int), cudaMemcpyHostToDevice, stream), "H2D new rows");
  // per node / per chain entry: the tree's arrays followed by the pseudo-blocks'
  auto ext = [&](const auto& base, const auto& add, auto** d) -> cudaError_t {
    using T = typename std::decay_t<decltype(base)>::value_type;
    std::vector<T> v(base.begin(), base.end());
    v.insert(v.end(), add.begin(), add.end());
    cudaError_t e = dalloc((void**)d, v.size() * sizeof(T));
    if (e != cudaSuccess) return e;
    // (from pageable memory: the call returns once v has been staged, so v may go out of scope)
    return cudaMemcpyAsync(*d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, stream);
  };
  std::vector<long long> zeros_ll(npb, 0);
  std::vector<int> zeros_i(npb, 0);
  int *d_m2, *d_row02, *d_k2, *d_P2, *d_choff2, *d_gs2, *d_chain2, *d_cpoff2;
  long long *d_goff2, *d_rioff2;
  ST_CUDA(ext(h_m, pm, &d_m2), "upload new nodes");
  ST_CUDA(ext(h_row0, prow0, &d_row02), "upload new nodes");
  ST_CUDA(ext(h_k, pk, &d_k2), "upload new nodes");
  ST_CUDA(ext(h_P, pP, &d_P2), "upload new nodes");
  ST_CUDA(ext(h_chain_off, pchoff, &d_choff2), "upload new nodes");
  ST_CUDA(ext(h_gs, zeros_i, &d_gs2), "upload new nodes");
  ST_CUDA(ext(h_goff, zeros_ll, &d_goff2), "upload new nodes");
  ST_CUDA(ext(h_rioff, prioff, &d_rioff2), "upload new nodes");
  ST_CUDA(ext(h_chain, pchain, &d_chain2), "upload new nodes");
  ST_CUDA(ext(h_chain_poff, pcpoff, &d_cpoff2), "upload new nodes");
  DevTree T2 = dt;
  T2.cx = d_cx2; T2.cy = d_cy2; T2.mvq = d_mvq2;
  T2.m = d_m2; T2.row0 = d_row02; T2.k = d_k2; T2.P = d_P2; T2.chain_off = d_choff2; T2.gs = d_gs2; T2.goff = d_goff2;
  T2.rioff = d_rioff2; T2.chain = d_chain2; T2.chain_poff = d_cpoff2;
  int *d_gslot0, *d_gnn, *d_cmvq;
  long long *d_lay2row, *d_perm;
  ST_CUDA(ext(std::vector<int>(), gslot0, &d_gslot0), "upload groups");
  ST_CUDA(ext(std::vector<int>(), gnn, &d_gnn), "upload groups");
  ST_CUDA(ext(std::vector<int>(), cmvq, &d_cmvq), "upload new rows");
  ST_CUDA(ext(std::vector<long long>(), std::vector<long long>(lay2row.begin(), lay2row.end()), &d_lay2row), "upload layout");
  ST_CUDA(ext(std::vector<long long>(), std::vector<long long>(perm.begin(), perm.end()), &d_perm), "upload perm");
  double* d_Xn = nullptr;
  if (R.X) {
    ST_CUDA(dalloc((void**)&d_Xn, (size_t)nn * p * sizeof(double)), "alloc");
    ST_CUDA(cudaMemcpyAsync(d_Xn, R.X, (size_t)nn * p * sizeof(double), cudaMemcpyHostToDevice, stream), "H2D X_new");
  }
  // samples of w staged in blocks of B (one 2D copy each), the node-ordered w_s, mean / sd, normals (from the store: every
  // sample is already on the device, one block of S); the draws of a sample go out from one of two staging slots of
  // 4 n_new doubles (w_new | y_new | mean | sd) while the next sample runs
  const int B = from_store ? S : (int)std::max<int64_t>(1, std::min<int64_t>(S, (256LL << 20) / (8 * n_all)));
  double *d_wblk = nullptr, *d_wnode, *d_mean, *d_sd, *d_acc, *d_zn = nullptr, *d_en = nullptr;
  if (!from_store) ST_CUDA(dalloc((void**)&d_wblk, (size_t)B * n_all * sizeof(double)), "alloc");
  ST_CUDA(dalloc((void**)&d_wnode, n_all * sizeof(double)), "alloc");
  ST_CUDA(dalloc((void**)&d_mean, nn * sizeof(double)), "alloc");
  ST_CUDA(dalloc((void**)&d_sd, nn * sizeof(double)), "alloc");
  ST_CUDA(dalloc((void**)&d_acc, 4 * nn * sizeof(double)), "alloc");
  if (PS.z) ST_CUDA(dalloc((void**)&d_zn, nn * sizeof(double)), "alloc");
  if (PS.eps) ST_CUDA(dalloc((void**)&d_en, nn * sizeof(double)), "alloc");
  double* const hout[4] = {out.w_new, out.y_new, out.mean, out.sd};
  CopyOut co(stream, copy_stream, err);
  int rc = co.open({hout[0], hout[1], hout[2], hout[3]}, (size_t)nn * S * sizeof(double), 2, 4 * (size_t)nn);
  if (rc) return rc;

  int last_ref = 0;
  while (last_ref < (int)levels.size() && levels[last_ref].is_ref) last_ref++;
  dvec built;  // theta of the alter slot's BUILD (empty: none yet)
  std::vector<int> build_of(S);  // the BUILD each sample is predicted from
  int* d_bfail;                  // failed factorisations of each BUILD
  ST_CUDA(dalloc((void**)&d_bfail, (size_t)S * sizeof(int)), "alloc");
  const int alt = phys(1);
  int si = 1, sb = (int)n_all;
  const double* wsrc = from_store ? PS.w : d_wblk;
  for (int j = 0; j < S; j++) {
    if (!from_store && j % B == 0) {
      const int nb = std::min(B, S - j);
      if (rmaj) {
        ST_CUDA(cudaMemcpy2DAsync(d_wblk, nb * sizeof(double), PS.w + j, PS.w_row_stride * sizeof(double), nb * sizeof(double), n_all,
                                  cudaMemcpyHostToDevice, stream), "H2D w samples");
        si = nb; sb = 1;
      } else {
        ST_CUDA(cudaMemcpy2DAsync(d_wblk, n_all * sizeof(double), PS.w + (size_t)j * PS.w_sample_stride, PS.w_sample_stride * sizeof(double),
                                  n_all * sizeof(double), nb, cudaMemcpyHostToDevice, stream), "H2D w samples");
        si = 1; sb = (int)n_all;
      }
    }
    const double* th = PS.theta + (size_t)j * npar;
    if (built.empty() || std::memcmp(built.data(), th, npar * sizeof(double)) != 0) {
      ThetaPack pkk;
      std::string e;
      pkk.n = npar;
      std::copy(th, th + npar, pkk.theta);
      if (!make_covtab(th, npar, q, pkk.tab, e)) { err = "predict_new: sample " + std::to_string(j) + ": " + e; return 1; }
      ST_CUDA(launch_chain_set_theta(d_mc, 1, pkk, stream), "chain_set_theta_kernel");
      deferred_[alt] = false;  // (from here on the slot holds the reference levels of this theta only)
      alter_scratch = true;
      rc = launch_build_levels(1, 0, last_ref, true, stream);
      if (rc) return rc;
      // the BUILD's failure count, kept per BUILD; the counter is the chain's and starts from zero again
      ST_CUDA(cudaMemcpyAsync(d_bfail + out.n_builds, d_fail, sizeof(int), cudaMemcpyDeviceToDevice, stream), "D2D fail");
      ST_CUDA(cudaMemsetAsync(d_fail, 0, sizeof(int), stream), "memset");
      built.assign(th, th + npar);
      out.n_builds++;
    }
    build_of[j] = (int)out.n_builds - 1;
    ST_CUDA(launch_gather_sample(wsrc, si, sb, j % B, d_perm, d_wnode, n_all, stream), "gather_sample_kernel");
    for (const LevelInfo::BuildLaunch& L : launches)
      ST_CUDA(launch_build(3, T2, dslots, 1, d_mean, d_sd, 0, d_gslot0 + L.grp0, d_gnn + L.grp0, L.ngrp, d_wnode, d_fail + 2, L.ns, 0,
                           L.smem, stream, L.threads),
              "build_level_kernel(predict_new)");
    if (d_zn) ST_CUDA(cudaMemcpyAsync(d_zn, PS.z + (size_t)j * nn, nn * sizeof(double), cudaMemcpyHostToDevice, stream), "H2D z");
    if (d_en) ST_CUDA(cudaMemcpyAsync(d_en, PS.eps + (size_t)j * nn, nn * sizeof(double), cudaMemcpyHostToDevice, stream), "H2D eps");
    const int r = j & 1;
    double* stage = co.buffer(r);
    if (!stage) return 2;
    PredDrawPack pack{};
    for (int jq = 0; jq < q; jq++) {
      for (int a = 0; a < p; a++) pack.beta[a + jq * p] = PS.beta[a + (size_t)j * p + (size_t)jq * p * S];
      pack.sdtau[jq] = std::sqrt(PS.tausq[jq + (size_t)j * q]);
    }
    double* dsrc[4] = {keep_draws ? store.get(2).d + (size_t)j * nn : stage, keep_draws ? store.get(3).d + (size_t)j * nn : stage + nn,
                       stage + 2 * nn, stage + 3 * nn};
    ST_CUDA(launch_predict_draw(nn, d_lay2row, d_cmvq, d_Xn, p, d_mean, d_sd, pack, PS.seed, j, d_zn, d_en, dsrc[0], dsrc[1],
                                dsrc[2], dsrc[3], d_acc, stream),
            "predict_draw_kernel");
    n_launches += 2 + (double)launches.size();
    double* hdst[4];
    for (int c = 0; c < 4; c++) hdst[c] = hout[c] ? hout[c] + (size_t)j * nn : nullptr;
    rc = co.send(r, hdst, dsrc, 4, nn);
    if (rc) return rc;
  }
  double* hm[4] = {out.w_mean, out.w_sd, out.y_mean, out.y_sd};
  if (hm[0] || hm[1] || hm[2] || hm[3]) {
    double* d_mom = d_wblk;  // (free once the last gather has run: 4 nn doubles fit when nn <= B n_all / 4, else its own)
    if (!d_wblk || 4 * nn > (int64_t)B * n_all) ST_CUDA(dalloc((void**)&d_mom, 4 * nn * sizeof(double)), "alloc");
    ST_CUDA(launch_predict_moments(nn, S, d_acc, d_mom, stream), "predict_moments_kernel");
    for (int c = 0; c < 4; c++)
      if (hm[c]) ST_CUDA(cudaMemcpyAsync(hm[c], d_mom + (size_t)c * nn, nn * sizeof(double), cudaMemcpyDeviceToHost, stream), "D2H moments");
  }
  std::vector<int> bfail(out.n_builds);
  ST_CUDA(cudaMemcpyAsync(bfail.data(), d_bfail, bfail.size() * sizeof(int), cudaMemcpyDeviceToHost, stream), "D2H fail");
  // the one synchronisation
  ST_CUDA(cudaStreamSynchronize(stream), "sync");
  rc = co.finish();
  if (rc) return rc;
  // a theta whose covariance is not positive definite on some reference block: the chain would have rejected it, and its
  // draws are not draws of the model (the factor rows of that block are zeroed)
  for (int j = 0; j < S; j++)
    if (bfail[build_of[j]] != 0) {
      err = "predict_new: theta of sample " + std::to_string(j) + ": a reference-level Cholesky factorisation failed (covariance not positive definite)";
      return 3;
    }
  if (keep_draws) store.commit(DrawStore::kPrediction, nn, S);
  return 0;
}

}  // namespace st
