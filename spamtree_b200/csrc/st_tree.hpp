// st_tree.hpp — host-side DAG construction (see st_tree.cpp)
#pragma once
#include <string>

#include "st_common.hpp"

namespace st {

void kthresholds(const double* x, int64_t n, int k, double* res);
void part_axis_parallel_lmt(const double* coords, int64_t n, int d, const double* thr, const int64_t* thr_ptr,
                            double* out);
void number_revalue(const int64_t* orig, int64_t nr, int nc, const int64_t* from_val, const int64_t* to_val,
                    int64_t nfrom, int64_t* out);
void make_edges(const double* parchimat, int64_t nr, int L, const int64_t* non_empty_blocks, int64_t n_ne,
                const int64_t* res_is_ref, bool limited, CSR& parents, CSR& children, int64_t& n_blocks);

// rows of the last loop level: the 1-NN targets of leftover, missing and attached rows
struct NNTargets {
  dvec x, y;
  ivec mv, block;  // 1-based outcome, 1-based block name
};
void nn_assign(const NNTargets& t, const double* qx, const double* qy, const int64_t* qmv, int64_t nq, bool same_margin,
               ivec& parent_block);

struct TreeResult {
  int64_t n_all = 0, n_blocks = 0, parchi_rows = 0;
  int parchi_cols = 0;
  ivec blocking, res, res_is_ref;
  dvec parchimat;  // parchi_rows x parchi_cols, NaN = NA
  CSR indexing, parents, children;
  dvec block_names, block_groups;
  // what attaching new rows needs (tree_attach)
  NNTargets last;
  bool cherrypick_same_margin = true;
  int n_loop_levels = 0;
};
bool make_tree(const double* coords, const double* y, const int64_t* mv_id, int64_t n_all, int cell_size, int K0,
               int K1, int start_level, int tree_depth, bool last_not_reference, bool cherrypick_same_margin,
               bool cherrypick_group_locations, uint64_t seed, TreeResult& T, std::string& err);
// coords_new: n_new x 2 column-major, mv_new 1-based.  group[i]: 0-based group of new row i; parents: per group, 0-based
// block ids, root first
bool tree_attach(const TreeResult& T, const double* coords_new, const int64_t* mv_new, int64_t n_new, bool limited, ivec& group,
                 CSR& parents, std::string& err);

}  // namespace st
