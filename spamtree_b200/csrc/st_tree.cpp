// st_tree.cpp — host-side DAG construction (integer / compare logic; results must match the reference bit-exactly).
//
// Re-designs of tree_dep.cpp (kthresholds :16-27, part_axis_parallel_lmt :42-67, make_edges :75-130,
// make_edges_limited :133-186, number_revalue :240-259) with the same outputs but O(n log n) data movement instead of
// the reference's repeated full scans, plus a deterministic stand-in for R's make_tree() (R/make_tree.R:1-420,
// R/axis_parallel.R:1-41) so that the C++ boundary inputs can be produced without R.
#include "st_tree.hpp"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <limits>
#include <numeric>
#include <string>
#include <unordered_map>
#include <unordered_set>

namespace st {

// tree_dep.cpp:16-27: res(i-1) = Q1-th order statistic with Q1 = i*n/k in unsigned 32-bit arithmetic.  The reference
// runs nth_element k-1 times on the same buffer; the value at an order statistic does not depend on that history, so one
// sort gives identical doubles.
void kthresholds(const double* x, int64_t n, int k, double* res) {
  if (k <= 1) return;
  dvec xs(x, x + n);
  std::sort(xs.begin(), xs.end());
  for (unsigned int i = 1; i < (unsigned int)k; i++) {
    unsigned int Q1 = (unsigned int)(i * (unsigned int)n / (unsigned int)k);
    res[i - 1] = xs[Q1];
  }
}

// the same order statistics from an array that is already sorted (make_tree asks for them at every level of both grids)
static void kthresholds_sorted(const dvec& xs, int k, double* res) {
  const int64_t n = (int64_t)xs.size();
  for (unsigned int i = 1; i < (unsigned int)k; i++) {
    unsigned int Q1 = (unsigned int)(i * (unsigned int)n / (unsigned int)k);
    res[i - 1] = xs[Q1];
  }
}

// tree_dep.cpp:42-55: 1 + #{j : x >= thresholds(j)}
static inline int count_over(double x, const double* thr, int64_t nt, bool sorted) {
  if (sorted) return 1 + (int)(std::upper_bound(thr, thr + nt, x) - thr);
  int over = 1;
  for (int64_t j = 0; j < nt; j++)
    if (x >= thr[j]) over++;
  return over;
}
void part_axis_parallel_lmt(const double* coords, int64_t n, int d, const double* thr, const int64_t* thr_ptr,
                            double* out) {
  for (int j = 0; j < d; j++) {
    const double* t = thr + thr_ptr[j];
    const int64_t nt = thr_ptr[j + 1] - thr_ptr[j];
    bool sorted = std::is_sorted(t, t + nt);
    for (int64_t i = 0; i < n; i++) {
      const double x = coords[i + (size_t)j * n];
      // NaN compares false everywhere in the reference loop -> 1
      out[i + (size_t)j * n] = std::isnan(x) ? 1 : count_over(x, t, nt, sorted);
    }
  }
}

// tree_dep.cpp:240-259: first matching from_val wins; results above max(to_val) become 0
void number_revalue(const int64_t* orig, int64_t nr, int nc, const int64_t* from_val, const int64_t* to_val,
                    int64_t nfrom, int64_t* out) {
  std::unordered_map<int64_t, int64_t> first;
  first.reserve((size_t)nfrom * 2);
  int64_t maxval = nfrom > 0 ? to_val[0] : 0;
  for (int64_t j = 0; j < nfrom; j++) {
    first.emplace(from_val[j], to_val[j]);  // emplace keeps the first occurrence
    maxval = std::max(maxval, to_val[j]);
  }
  for (int64_t e = 0; e < nr * nc; e++) {
    auto it = first.find(orig[e]);
    int64_t v = (it == first.end()) ? orig[e] : it->second;
    if (v > maxval) v = 0;
    out[e] = v;
  }
}

// tree_dep.cpp:75-186.  Blocks of one level are found by sorting the rows of that column once; the parent / child
// sets of a block are the sorted unique finite names in the selected columns of its rows.
void make_edges(const double* parchimat, int64_t nr, int L, const int64_t* non_empty_blocks, int64_t n_ne,
                const int64_t* res_is_ref, bool limited, CSR& parents, CSR& children, int64_t& n_blocks) {
  n_blocks = 0;
  for (int64_t i = 0; i < nr; i++) {
    const double v = parchimat[i + (size_t)(L - 1) * nr];
    if (std::isfinite(v)) n_blocks = std::max(n_blocks, (int64_t)v);
  }
  std::vector<ivec> par(n_blocks), chi(n_blocks);
  std::vector<char> is_ne(n_blocks + 1, 0);
  for (int64_t i = 0; i < n_ne; i++)
    if (non_empty_blocks[i] >= 1 && non_empty_blocks[i] <= n_blocks) is_ne[non_empty_blocks[i]] = 1;
  ivec reference_res;
  for (int l = 0; l < L; l++)
    if (res_is_ref[l] == 1) reference_res.push_back(l);

  std::vector<int64_t> order(nr);
  for (int lev = 0; lev < L; lev++) {
    const double* col = parchimat + (size_t)lev * nr;
    int64_t nfin = 0;
    for (int64_t i = 0; i < nr; i++)
      if (std::isfinite(col[i])) order[nfin++] = i;
    std::sort(order.begin(), order.begin() + nfin, [&](int64_t a, int64_t b) { return col[a] < col[b]; });
    ivec colselect;
    if (lev > 0) {
      if (!reference_res.empty()) {
        for (int64_t r : reference_res)
          if (r < lev) colselect.push_back(r);
      } else {
        for (int c = 0; c < lev; c++) colselect.push_back(c);
      }
      if (limited && !colselect.empty()) colselect.assign(1, colselect.back());
    }
    const bool gives_children = (res_is_ref[lev] == 1) && (lev < L - 1);
    const int last_child_col = limited ? lev + 1 : L - 1;
    for (int64_t s = 0; s < nfin;) {
      int64_t e = s;
      while (e < nfin && col[order[e]] == col[order[s]]) e++;
      const int64_t u = (int64_t)col[order[s]] - 1;
      if (u >= 0 && u < n_blocks) {
        ivec vals;
        if (gives_children) {
          for (int c = lev + 1; c <= last_child_col; c++)
            for (int64_t k = s; k < e; k++) {
              const double v = parchimat[order[k] + (size_t)c * nr];
              if (std::isfinite(v) && (int64_t)v >= 1 && (int64_t)v <= n_blocks && is_ne[(int64_t)v])
                vals.push_back((int64_t)v - 1);
            }
          std::sort(vals.begin(), vals.end());
          vals.erase(std::unique(vals.begin(), vals.end()), vals.end());
          chi[u] = vals;
        }
        if (lev > 0) {
          vals.clear();
          for (int64_t c : colselect)
            for (int64_t k = s; k < e; k++) {
              const double v = parchimat[order[k] + (size_t)c * nr];
              if (std::isfinite(v)) vals.push_back((int64_t)v - 1);
            }
          std::sort(vals.begin(), vals.end());
          vals.erase(std::unique(vals.begin(), vals.end()), vals.end());
          par[u] = vals;
        }
      }
      s = e;
    }
  }
  parents.ptr.assign(n_blocks + 1, 0);
  children.ptr.assign(n_blocks + 1, 0);
  parents.idx.clear();
  children.idx.clear();
  for (int64_t i = 0; i < n_blocks; i++) {
    parents.idx.insert(parents.idx.end(), par[i].begin(), par[i].end());
    children.idx.insert(children.idx.end(), chi[i].begin(), chi[i].end());
    parents.ptr[i + 1] = (int64_t)parents.idx.size();
    children.ptr[i + 1] = (int64_t)children.idx.size();
  }
}

// ------------------------------------------------------------------------------------------------------------------
// make_tree stand-in
namespace {

inline uint64_t mix64(uint64_t x) {
  uint64_t z = x + 0x9E3779B97F4A7C15ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}

// R/axis_parallel.R:9-23: per-axis cell ids become factors whose levels sort as CHARACTER strings; the block id is the
// rank of the (axis1, axis2) combination among the combinations present, axis 1 varying fastest.
ivec axis_parallel_block(const std::vector<int>& c1, const std::vector<int>& c2) {
  const size_t n = c1.size();
  ivec block(n, 1);
  if (n <= 1) return block;
  auto lex_rank = [](const std::vector<int>& c, std::vector<int>& rank_of, int& nlev) {
    int mx = 0;
    for (int v : c) mx = std::max(mx, v);
    std::vector<char> present(mx + 1, 0);
    for (int v : c) present[v] = 1;
    std::vector<std::pair<std::string, int>> lv;
    for (int v = 0; v <= mx; v++)
      if (present[v]) lv.emplace_back(std::to_string(v), v);
    std::sort(lv.begin(), lv.end());
    rank_of.assign(mx + 1, -1);
    for (size_t i = 0; i < lv.size(); i++) rank_of[lv[i].second] = (int)i;
    nlev = (int)lv.size();
  };
  std::vector<int> r1, r2;
  int n1 = 0, n2 = 0;
  lex_rank(c1, r1, n1);
  lex_rank(c2, r2, n2);
  ivec comb(n);
  for (size_t i = 0; i < n; i++) comb[i] = (int64_t)r1[c1[i]] + (int64_t)n1 * r2[c2[i]];
  ivec present(comb);
  std::sort(present.begin(), present.end());
  present.erase(std::unique(present.begin(), present.end()), present.end());
  for (size_t i = 0; i < n; i++)
    block[i] = 1 + (int64_t)(std::lower_bound(present.begin(), present.end(), comb[i]) - present.begin());
  return block;
}

// exact 1-NN on a bucket grid; ties resolved towards the smaller target position
struct NNGrid {
  int G = 1;
  double x0 = 0, y0 = 0, sx = 1, sy = 1;
  const double *tx = nullptr, *ty = nullptr;
  ivec cell_ptr, cell_idx;
  void build(const double* tx_, const double* ty_, int64_t nt) {
    tx = tx_;
    ty = ty_;
    double x1 = -std::numeric_limits<double>::infinity(), y1 = x1;
    x0 = y0 = std::numeric_limits<double>::infinity();
    for (int64_t i = 0; i < nt; i++) {
      x0 = std::min(x0, tx[i]); x1 = std::max(x1, tx[i]);
      y0 = std::min(y0, ty[i]); y1 = std::max(y1, ty[i]);
    }
    G = std::max(1, (int)std::sqrt((double)nt / 2.0));
    sx = (x1 > x0) ? G / (x1 - x0) : 1.0;
    sy = (y1 > y0) ? G / (y1 - y0) : 1.0;
    cell_ptr.assign((size_t)G * G + 1, 0);
    ivec cell_of(nt);
    for (int64_t i = 0; i < nt; i++) {
      cell_of[i] = cx(tx[i]) + (int64_t)G * cy(ty[i]);
      cell_ptr[cell_of[i] + 1]++;
    }
    for (size_t c = 0; c < (size_t)G * G; c++) cell_ptr[c + 1] += cell_ptr[c];
    cell_idx.resize(nt);
    ivec fill(cell_ptr.begin(), cell_ptr.end() - 1);
    for (int64_t i = 0; i < nt; i++) cell_idx[fill[cell_of[i]]++] = i;
  }
  int cx(double x) const { return std::min(G - 1, std::max(0, (int)((x - x0) * sx))); }
  int cy(double y) const { return std::min(G - 1, std::max(0, (int)((y - y0) * sy))); }
  int64_t query(double qx, double qy) const {
    const int c0 = cx(qx), r0 = cy(qy);
    double best = std::numeric_limits<double>::infinity();
    int64_t bi = -1;
    const double wx = 1.0 / sx, wy = 1.0 / sy;
    for (int ring = 0; ring <= G; ring++) {
      // the ring-th shell of cells around (c0, r0)
      for (int r = r0 - ring; r <= r0 + ring; r++) {
        if (r < 0 || r >= G) continue;
        const bool edge_row = (r == r0 - ring || r == r0 + ring);
        for (int c = c0 - ring; c <= c0 + ring; c += (edge_row ? 1 : 2 * ring > 0 ? 2 * ring : 1)) {
          if (c < 0 || c >= G) continue;
          const int64_t cell = c + (int64_t)G * r;
          for (int64_t k = cell_ptr[cell]; k < cell_ptr[cell + 1]; k++) {
            const int64_t t = cell_idx[k];
            const double dx = tx[t] - qx, dy = ty[t] - qy, d2 = dx * dx + dy * dy;
            if (d2 < best || (d2 == best && t < bi)) { best = d2; bi = t; }
          }
        }
      }
      if (bi >= 0) {
        // every target outside the searched square is at least `lim` away (sides already at the grid edge do not count)
        double lim = std::numeric_limits<double>::infinity();
        if (c0 - ring > 0) lim = std::min(lim, qx - (x0 + (c0 - ring) * wx));
        if (c0 + ring < G - 1) lim = std::min(lim, (x0 + (c0 + ring + 1) * wx) - qx);
        if (r0 - ring > 0) lim = std::min(lim, qy - (y0 + (r0 - ring) * wy));
        if (r0 + ring < G - 1) lim = std::min(lim, (y0 + (r0 + ring + 1) * wy) - qy);
        lim -= 1e-9 * (wx + wy);  // guard against rounding in the cell assignment
        if (lim > 0 && lim * lim >= best) break;
      }
    }
    return bi;
  }
};

}  // namespace

// per-margin 1-NN targets among rows of the last loop level (:218, :322): parent_block[i] = block of the target nearest to
// query i, among the targets of the query's own margin when same_margin is set (any margin when that one has none)
void nn_assign(const NNTargets& t, const double* qx, const double* qy, const int64_t* qmv, int64_t nq, bool same_margin,
               ivec& parent_block) {
  parent_block.assign(nq, 0);
  std::vector<int64_t> margins;
  if (same_margin) {
    margins.assign(qmv, qmv + nq);
    std::sort(margins.begin(), margins.end());
    margins.erase(std::unique(margins.begin(), margins.end()), margins.end());
  } else {
    margins.push_back(-1);
  }
  const int64_t nt = (int64_t)t.x.size();
  for (int64_t vv : margins) {
    ivec tsel;
    for (int64_t r = 0; r < nt; r++)
      if (vv < 0 || t.mv[r] == vv) tsel.push_back(r);
    if (tsel.empty())  // FNN would stop here; fall back to any margin
      for (int64_t r = 0; r < nt; r++) tsel.push_back(r);
    dvec tx(tsel.size()), ty(tsel.size());
    for (size_t i = 0; i < tsel.size(); i++) { tx[i] = t.x[tsel[i]]; ty[i] = t.y[tsel[i]]; }
    NNGrid g;
    g.build(tx.data(), ty.data(), (int64_t)tsel.size());
    for (int64_t qi = 0; qi < nq; qi++) {
      if (vv >= 0 && qmv[qi] != vv) continue;
      parent_block[qi] = t.block[tsel[g.query(qx[qi], qy[qi])]];
    }
  }
}

// R/make_tree.R:1-420 (structure) + the tail of spamtree() that turns it into the boundary inputs
// (R/spamtree_fit.R:288-324).
bool make_tree(const double* coords, const double* y, const int64_t* mv_id, int64_t n_all, int cell_size, int K0,
               int K1, int start_level, int tree_depth, bool last_not_reference, bool cherrypick_same_margin,
               bool cherrypick_group_locations, uint64_t seed, TreeResult& T, std::string& err) {
  const double* X0 = coords;
  const double* X1 = coords + n_all;
  const int K[2] = {K0, K1};
  // ST_PROFILE_TREE=1: wall-clock per section on stderr (development aid)
  static const bool prof = getenv("ST_PROFILE_TREE") != nullptr;
  auto tlast = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!prof) return;
    const auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[tree profile] %-28s %.3f s\n", what, std::chrono::duration<double>(now - tlast).count());
    tlast = now;
  };
  const int axis_size = (int)std::lround(std::pow((double)cell_size, 0.5));  // R/spamtree_fit.R:229-233
  const double max_res = (tree_depth <= 0) ? std::numeric_limits<double>::infinity() : (double)(start_level + tree_depth);

  ivec avail, missing;
  for (int64_t i = 0; i < n_all; i++) (std::isnan(y[i]) ? missing : avail).push_back(i);
  const int64_t na = (int64_t)avail.size();
  if (na == 0) { err = "no observed rows"; return false; }
  dvec a0(na), a1(na);
  for (int64_t i = 0; i < na; i++) { a0[i] = X0[avail[i]]; a1[i] = X1[avail[i]]; }
  dvec s0(a0), s1(a1);  // sorted once: every grid of every level takes its quantiles from them
  std::sort(s0.begin(), s0.end());
  std::sort(s1.begin(), s1.end());

  T.n_all = n_all;
  T.blocking.assign(n_all, 0);
  T.res.assign(n_all, 0);
  T.res_is_ref.clear();

  ivec cx = avail;  // observed rows not yet placed
  // block-grid cell (per axis) of every observed row at every loop level, and the block name living in each cell
  std::vector<std::vector<int>> lvl_c0, lvl_c1;              // per level, per avail position
  std::vector<std::vector<int64_t>> lvl_cell2block;  // per level: cell key -> block name (0: no row placed there), dense
  std::vector<int> lvl_res;
  int64_t max_block_number = 0;
  int res = start_level + 1, res_ix = 1;
  ivec last_level_rows;  // rows placed at the last loop level

  auto cells_of = [&](const ivec& rows, const dvec& t0, const dvec& t1, std::vector<int>& c0, std::vector<int>& c1) {
    c0.resize(rows.size());
    c1.resize(rows.size());
    for (size_t i = 0; i < rows.size(); i++) {
      c0[i] = count_over(X0[rows[i]], t0.data(), (int64_t)t0.size(), true);
      c1[i] = count_over(X1[rows[i]], t1.data(), (int64_t)t1.size(), true);
    }
  };

  while ((double)res <= max_res && !cx.empty()) {
    // knot grid: quantiles of ALL observed coordinates (R/make_tree.R:79-80)
    const double kk0 = (double)axis_size * std::pow((double)K[0], res - 1), kk1 = (double)axis_size * std::pow((double)K[1], res - 1);
    ivec picked;
    const double grid_size = kk0 * kk1;
    if (grid_size < (double)cx.size()) {  // :84
      dvec t0((size_t)kk0 - 1), t1((size_t)kk1 - 1);
      kthresholds_sorted(s0, (int)kk0, t0.data());
      kthresholds_sorted(s1, (int)kk1, t1.data());
      std::vector<int> c0, c1;
      cells_of(cx, t0, t1, c0, c1);
      // one row per non-empty knot cell: smallest mix64(ix ^ seed)  (stand-in for sample(), :92).  mix64 is a bijection, so
      // the winner of a cell is unique: one pass finds it (no sort of the unplaced rows by cell)
      const int64_t kstride = (int64_t)(kk1 + 1);
      auto key = [&](size_t i) { return (int64_t)c0[i] * kstride + c1[i]; };
      const int64_t nkeys = ((int64_t)kk0 + 1) * kstride;
      const bool dense = nkeys <= 8 * (int64_t)cx.size() + 4096;
      std::vector<int64_t> win_dense;                 // cell -> position in cx of its winner (-1: empty)
      std::unordered_map<int64_t, int64_t> win_map;
      if (dense) win_dense.assign((size_t)nkeys, -1);
      std::vector<uint64_t> mixv(cx.size());
      for (size_t i = 0; i < cx.size(); i++) {
        mixv[i] = mix64((uint64_t)cx[i] ^ seed);
        const int64_t k = key(i);
        if (dense) {
          int64_t& wv = win_dense[(size_t)k];
          if (wv < 0 || mixv[i] < mixv[(size_t)wv]) wv = (int64_t)i;
        } else {
          auto it = win_map.find(k);
          if (it == win_map.end()) win_map.emplace(k, (int64_t)i);
          else if (mixv[i] < mixv[(size_t)it->second]) it->second = (int64_t)i;
        }
      }
      auto winner_of = [&](int64_t k) { return dense ? win_dense[(size_t)k] : win_map.find(k)->second; };
      for (size_t i = 0; i < cx.size(); i++) {
        const int64_t wv = winner_of(key(i));
        if ((int64_t)i == wv) { picked.push_back(cx[i]); continue; }
        if (cherrypick_group_locations) {  // :94-99: every unplaced row at the winner's location comes along
          const int64_t r = cx[(size_t)wv], r2 = cx[i];
          if (X0[r2] == X0[r] && X1[r2] == X1[r]) picked.push_back(r2);
        }
      }
      std::sort(picked.begin(), picked.end());
      lap("  knots: pick one row per cell");
    } else {
      picked = cx;  // :106-108
    }
    // block grid (:118) and block names of the picked rows (:121-130)
    const int kb0 = (int)std::pow((double)K[0], res - 1), kb1 = (int)std::pow((double)K[1], res - 1);
    dvec tb0(std::max(0, kb0 - 1)), tb1(std::max(0, kb1 - 1));
    kthresholds_sorted(s0, kb0, tb0.data());
    kthresholds_sorted(s1, kb1, tb1.data());
    std::vector<int> pc0, pc1;
    cells_of(picked, tb0, tb1, pc0, pc1);
    ivec pb = axis_parallel_block(pc0, pc1);
    lap("  block grid + names");
    std::vector<int64_t> cell2block((size_t)(kb0 + 1) * (size_t)(kb1 + 1), 0);
    int64_t new_max = max_block_number;
    for (size_t i = 0; i < picked.size(); i++) {
      const int64_t b = max_block_number + pb[i];
      T.blocking[picked[i]] = b;
      T.res[picked[i]] = res;
      cell2block[(size_t)pc0[i] * (size_t)(kb1 + 1) + pc1[i]] = b;
      new_max = std::max(new_max, b);
    }
    max_block_number = new_max;
    // remove picked rows from cx (:137)
    {
      ivec rest;
      rest.reserve(cx.size() - picked.size());
      std::set_difference(cx.begin(), cx.end(), picked.begin(), picked.end(), std::back_inserter(rest));
      cx.swap(rest);
    }
    // keep track of every observed row's block-grid cell at this level (:141-149)
    std::vector<int> ac0, ac1;
    cells_of(avail, tb0, tb1, ac0, ac1);
    lvl_c0.push_back(ac0);
    lvl_c1.push_back(ac1);
    lvl_cell2block.push_back(std::move(cell2block));
    lvl_res.push_back(kb1 + 1);
    last_level_rows = picked;
    lap("  cells of all rows");
    T.res_is_ref.push_back(1);
    res++;
    res_ix++;
  }
  const int nlev = (int)lvl_c0.size();
  if (last_not_reference && ((double)res < max_res) && nlev > 0) T.res_is_ref[nlev - 1] = 0;  // :162-165

  // parchi_map (:175-208): one row per distinct root-to-leaf chain of block-grid cells over placed rows; a cell is
  // translated to the block name that lives in it (NA when no row was placed there at that level)
  std::vector<char> placed(n_all, 0);
  for (int64_t i = 0; i < n_all; i++) placed[i] = T.blocking[i] > 0;
  std::vector<ivec> chains;
  {
    // (most rows share their chain with the other rows of their leaf cell: distinct chains are collected by hashing first,
    // only those are sorted)
    std::vector<std::vector<int64_t>> rows;
    struct VecHash {
      size_t operator()(const ivec& v) const {
        uint64_t h = 0x9E3779B97F4A7C15ULL;
        for (int64_t x : v) h = mix64(h ^ (uint64_t)x);
        return (size_t)h;
      }
    };
    std::unordered_set<ivec, VecHash> seen_chains;
    ivec ch(nlev);
    for (int64_t ai = 0; ai < na; ai++) {
      if (!placed[avail[ai]]) continue;
      for (int l = 0; l < nlev; l++) ch[l] = lvl_cell2block[l][(size_t)lvl_c0[l][ai] * (size_t)lvl_res[l] + lvl_c1[l][ai]];
      if (seen_chains.insert(ch).second) rows.push_back(ch);
    }
    // arrange(): ascending by columns, NA (0) last; then unique
    auto na_last = [](int64_t v) { return v == 0 ? std::numeric_limits<int64_t>::max() : v; };
    std::sort(rows.begin(), rows.end(), [&](const ivec& a, const ivec& b) {
      for (size_t l = 0; l < a.size(); l++)
        if (a[l] != b[l]) return na_last(a[l]) < na_last(b[l]);
      return false;
    });
    rows.erase(std::unique(rows.begin(), rows.end()), rows.end());
    chains.swap(rows);
  }
  lap("chains (parchi_map)");
  int ncols = nlev;
  max_block_number = 0;
  for (int64_t i = 0; i < n_all; i++) max_block_number = std::max(max_block_number, T.blocking[i]);
  const int64_t loop_max_res = nlev > 0 ? (start_level + nlev) : start_level;

  // the 1-NN targets: rows of the last loop level (kept with the tree, st_tree_attach attaches new rows by the same rule)
  T.last = NNTargets();
  for (int64_t r : last_level_rows) {
    T.last.x.push_back(X0[r]); T.last.y.push_back(X1[r]); T.last.mv.push_back(mv_id[r]); T.last.block.push_back(T.blocking[r]);
  }
  T.cherrypick_same_margin = cherrypick_same_margin;
  T.n_loop_levels = nlev;
  auto nn_rows = [&](const ivec& queries, ivec& parent_block) {
    dvec qx(queries.size()), qy(queries.size());
    ivec qmv(queries.size());
    for (size_t i = 0; i < queries.size(); i++) { qx[i] = X0[queries[i]]; qy[i] = X1[queries[i]]; qmv[i] = mv_id[queries[i]]; }
    nn_assign(T.last, qx.data(), qy.data(), qmv.data(), (int64_t)queries.size(), cherrypick_same_margin, parent_block);
  };
  // new block names: as.numeric(factor(parent block)) + max_block_number (:280, :385)
  auto rank_blocks = [&](const ivec& parent_block, ivec& newblock) {
    ivec u(parent_block);
    std::sort(u.begin(), u.end());
    u.erase(std::unique(u.begin(), u.end()), u.end());
    newblock.resize(parent_block.size());
    for (size_t i = 0; i < parent_block.size(); i++)
      newblock[i] = 1 + (int64_t)(std::lower_bound(u.begin(), u.end(), parent_block[i]) - u.begin()) + max_block_number;
  };
  // left_join of a (parent block -> new block) column onto the chains (:293-300, :400-410)
  auto join_column = [&](int parent_col, const ivec& parent_block, const ivec& newblock) {
    std::unordered_map<int64_t, int64_t> m;
    for (size_t i = 0; i < parent_block.size(); i++) m[parent_block[i]] = newblock[i];
    for (auto& ch : chains) {
      auto it = m.find(ch[parent_col]);
      ch.push_back(it == m.end() ? 0 : it->second);
    }
    ncols++;
  };

  int64_t cur_max_res = loop_max_res;
  if (!cx.empty()) {  // leftovers (:213-305)
    ivec pblock, nblock;
    nn_rows(cx, pblock);
    rank_blocks(pblock, nblock);
    const int64_t res_left = loop_max_res + 1;
    for (size_t i = 0; i < cx.size(); i++) { T.blocking[cx[i]] = nblock[i]; T.res[cx[i]] = res_left; }
    join_column(nlev - 1, pblock, nblock);
    T.res_is_ref.push_back(0);
    for (int64_t b : nblock) max_block_number = std::max(max_block_number, b);
    cur_max_res = res_left;
  }
  lap("leftovers: 1-NN + join");
  if (T.res_is_ref.size() == 1) T.res_is_ref[0] = 1;  // :307-309
  if (!missing.empty()) {  // rows to predict (:317-413)
    ivec pblock, nblock;
    nn_rows(missing, pblock);
    rank_blocks(pblock, nblock);
    const int64_t res_miss = cur_max_res + 1;
    for (size_t i = 0; i < missing.size(); i++) { T.blocking[missing[i]] = nblock[i]; T.res[missing[i]] = res_miss; }
    join_column(nlev - 1, pblock, nblock);
    T.res_is_ref.push_back(0);
    for (int64_t b : nblock) max_block_number = std::max(max_block_number, b);
  }
  lap("missing rows: 1-NN + join");
  // parchi_map %>% unique()
  std::sort(chains.begin(), chains.end());
  chains.erase(std::unique(chains.begin(), chains.end()), chains.end());
  T.parchi_rows = (int64_t)chains.size();
  T.parchi_cols = ncols;
  T.parchimat.assign((size_t)T.parchi_rows * ncols, std::numeric_limits<double>::quiet_NaN());
  for (int64_t i = 0; i < T.parchi_rows; i++)
    for (int c = 0; c < ncols; c++)
      if (chains[i][c] > 0) T.parchimat[i + (size_t)c * T.parchi_rows] = (double)chains[i][c];

  // ---- tail of spamtree(): R/spamtree_fit.R:288-324
  const int64_t n_blocks = max_block_number;
  T.n_blocks = n_blocks;
  // non_empty_blocks: blocks with at least one observed row (:296-303)
  std::vector<char> ne(n_blocks + 1, 0);
  for (int64_t i = 0; i < n_all; i++)
    if (!std::isnan(y[i])) ne[T.blocking[i]] = 1;
  ivec non_empty;
  for (int64_t b = 1; b <= n_blocks; b++)
    if (ne[b]) non_empty.push_back(b);
  int64_t nb2 = 0;
  make_edges(T.parchimat.data(), T.parchi_rows, ncols, non_empty.data(), (int64_t)non_empty.size(), T.res_is_ref.data(),
             false, T.parents, T.children, nb2);
  lap("parchimat + make_edges");
  if (nb2 != n_blocks) {
    // make_edges sizes by max(last column) (tree_dep.cpp:80); pad so that every block name has an entry
    T.parents.ptr.resize(n_blocks + 1, T.parents.ptr.back());
    T.children.ptr.resize(n_blocks + 1, T.children.ptr.back());
  }
  // block_names: first appearance in row order (:290-292, :322); block_groups: level by block id (:323)
  T.block_names.clear();
  T.block_groups.assign(n_blocks, 0.0);
  std::vector<char> seen(n_blocks + 1, 0);
  for (int64_t i = 0; i < n_all; i++) {
    const int64_t b = T.blocking[i];
    if (!seen[b]) { seen[b] = 1; T.block_names.push_back((double)b); T.block_groups[b - 1] = (double)T.res[i]; }
  }
  if ((int64_t)T.block_names.size() != n_blocks) { err = "internal: block names are not contiguous"; return false; }
  // indexing = split(0:(n-1), blocking) (:324)
  T.indexing.ptr.assign(n_blocks + 1, 0);
  for (int64_t i = 0; i < n_all; i++) T.indexing.ptr[T.blocking[i]]++;
  for (int64_t b = 0; b < n_blocks; b++) T.indexing.ptr[b + 1] += T.indexing.ptr[b];
  T.indexing.idx.resize(n_all);
  ivec fill(T.indexing.ptr.begin(), T.indexing.ptr.end() - 1);
  for (int64_t i = 0; i < n_all; i++) T.indexing.idx[fill[T.blocking[i] - 1]++] = i;
  lap("names, groups, indexing");
  return true;
}

// New rows attached to a built tree by the rule that makes the prediction level of make_tree (:317-413): the nearest row of
// the last loop level names the parent block b, the rows of one b form one group (groups ordered by b, as rank_blocks
// numbers them), and a group's parents are what make_edges / make_edges_limited would give a block in a column appended
// to parchimat: the reference blocks on the chains through b, root first.
bool tree_attach(const TreeResult& T, const double* coords_new, const int64_t* mv_new, int64_t n_new, bool limited, ivec& group,
                 CSR& parents, std::string& err) {
  group.assign(n_new, 0);
  parents.ptr.assign(1, 0);
  parents.idx.clear();
  if (n_new == 0) return true;
  if (T.last.x.empty() || T.n_loop_levels < 1) { err = "the tree has no loop level to attach rows to"; return false; }
  for (int64_t i = 0; i < n_new; i++)
    if (!std::isfinite(coords_new[i]) || !std::isfinite(coords_new[i + n_new])) { err = "coords_new holds a non-finite value"; return false; }
  ivec pblock;
  nn_assign(T.last, coords_new, coords_new + n_new, mv_new, n_new, T.cherrypick_same_margin, pblock);
  ivec u(pblock);
  std::sort(u.begin(), u.end());
  u.erase(std::unique(u.begin(), u.end()), u.end());
  for (int64_t i = 0; i < n_new; i++) group[i] = (int64_t)(std::lower_bound(u.begin(), u.end(), pblock[i]) - u.begin());
  // make_edges' colselect for a column L = parchi_cols
  const int L = T.parchi_cols;
  const int64_t nr = T.parchi_rows;
  ivec colselect;
  for (int l = 0; l < L && l < (int)T.res_is_ref.size(); l++)
    if (T.res_is_ref[l] == 1) colselect.push_back(l);
  if (colselect.empty())
    for (int c = 0; c < L; c++) colselect.push_back(c);
  if (limited) colselect.assign(1, colselect.back());
  // the chain rows through each b (the column of the last loop level)
  const double* bcol = T.parchimat.data() + (size_t)(T.n_loop_levels - 1) * nr;
  std::vector<ivec> par(u.size());
  for (int64_t r = 0; r < nr; r++) {
    if (!std::isfinite(bcol[r])) continue;
    const auto it = std::lower_bound(u.begin(), u.end(), (int64_t)bcol[r]);
    if (it == u.end() || *it != (int64_t)bcol[r]) continue;
    ivec& vals = par[it - u.begin()];
    for (int64_t c : colselect) {
      const double v = T.parchimat[r + (size_t)c * nr];
      if (std::isfinite(v)) vals.push_back((int64_t)v - 1);
    }
  }
  for (auto& vals : par) {
    std::sort(vals.begin(), vals.end());
    vals.erase(std::unique(vals.begin(), vals.end()), vals.end());
    parents.idx.insert(parents.idx.end(), vals.begin(), vals.end());
    parents.ptr.push_back((int64_t)parents.idx.size());
  }
  return true;
}

}  // namespace st
