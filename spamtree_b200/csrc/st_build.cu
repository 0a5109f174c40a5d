// st_build.cu — build_level_kernel: BUILD of one tree level (get_loglik_comps_w_std, spamtree_model.cpp:834-998) and
// of the prediction blocks (predict_std, :1234-1358).
//
// One CTA per work group = a run of sibling blocks (they share their ancestor chain).  Per group, in shared memory:
//   1. K = K_{pa,u}: cross-covariance panel, one column per row of the group's blocks (Covariancef_inplace, :885)
//   2. Z = L^-1 K : the chain's inverse Cholesky factor L^-1 (Kxx_invchol of the parent, :882) is never stored as a
//                   matrix; its rows are the row blocks [G_a | -Ri_a] (sign flipped, tree_utils.cpp:204-206) that every
//                   ancestor a wrote when its own level was built.  16 rows at a time are staged with cp.async and
//                   multiplied into the panel in place, bottom rows first.
//   3. R = K_uu - Z'Z (= Kcc - H Kxc, :896-897), Ri = chol(R)^-1 (non-reference levels: diagonal only, :931-948)
//   4. Y' = Z Ri' in place, then G' = L^-T Y' (= (Ri H)', :887-888 without ever forming Kxx_inv): 16 columns of L^-1
//      at a time are staged; the accumulators go straight to global memory, and G w_pa is accumulated on the way
//   5. wcore = |Ri w_u - G w_pa|^2, logdet (:912-913, :966-968)
// All dense contractions are FP64 tensor-core MMAs (mma.sync m8n8k4): one warp owns 8 panel columns, so that the
// in-place updates need no inter-warp synchronisation, and reuses every B fragment for two m-tiles.
#include <cuda_pipeline.h>
#include <cuda_runtime.h>

#include <cstdint>

#include "st_device.cuh"
#include "st_kernels.cuh"

namespace st {

namespace {
constexpr int RS = kBuildRS, ST = kBuildST;
#ifndef ST_COV_ILP
#define ST_COV_ILP 4
#endif
constexpr int kCovIlp = ST_COV_ILP;  // covariance evaluations in flight per thread

// D(8x8) += A(8x4, row) * B(4x8, col); lane l holds A[l>>2][l&3], B[l&3][l>>2], D[l>>2][2*(l&3) + {0,1}]
__device__ __forceinline__ void dmma(double (&c)[2], double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}

// R (row-major, stride rs, lower triangle valid, m <= 32) <- chol(R)^-1 (lower; strict upper zeroed) by a PAIR of warps
// that work one pivot apart: role 0 factorises, role 1 inverts.  Both are right-looking and keep their operand in
// registers, one row (factor) / one column (inverse) per lane, rotated so that the active entry is always element 0 and
// the loops stay rolled.  Step j of the factorisation publishes column j of L (cb: 2 x 64 doubles, double-buffered, zero
// past row 31) and 1 / L_jj (dv: 32 doubles); the pair meets at the 64-thread named barrier `bar`; then the factorising
// warp applies its trailing update a[i] <- a[i+1] - l_i l_(j+1+i) while the inverting warp finalises x_j = acc[0] / L_jj,
// row j of L^-1, and pushes -L[r][j] x_j into the rows below.  The two latency chains (tools/microbench/chol_bench.cu:
// ~360 and ~340 cycles per pivot) overlap instead of adding up.  Returns false on a non-positive pivot (dpotrf info > 0);
// the result is meaningful in the factorising warp only.
__device__ __noinline__ bool pair_chol_inv32(double* R, int m, int rs, double* cb, double* dv, int lane, int role, int bar) {
  bool ok = true;
  if (role == 0) {
    double a[32];
#pragma unroll
    for (int j = 0; j < 32; j++) a[j] = (lane < m && j <= lane) ? R[lane * rs + j] : 0.0;
    cb[32 + lane] = 0.0;
    cb[96 + lane] = 0.0;
    for (int j = 0; j < m; j++) {
      double d = __shfl_sync(0xffffffffu, a[0], j);
      if (!(d > 0.0) || !isfinite(d)) { ok = false; d = 1.0; }
      const double inv = rsqrt(d), sd = d * inv;
      const double l = (lane == j) ? sd : ((lane > j) ? a[0] * inv : 0.0);
      double* c = cb + (j & 1) * 64;
      c[lane] = l;
      if (lane == 0) dv[j] = inv;
      asm volatile("bar.sync %0, 64;" ::"r"(bar) : "memory");
      const double* cj = c + j + 1;  // l of rows j+1 ..; entries past row 31 are zero
#pragma unroll
      for (int i = 0; i < 31; i++) a[i] = fma(-l, cj[i], a[i + 1]);
      a[31] = 0.0;
    }
  } else {
    double acc[32];
#pragma unroll
    for (int i = 0; i < 32; i++) acc[i] = (i == lane) ? 1.0 : 0.0;
    for (int k = 0; k < m; k++) {
      asm volatile("bar.sync %0, 64;" ::"r"(bar) : "memory");
      const double x = acc[0] * dv[k];
      const double* cj = cb + (k & 1) * 64 + k + 1;
#pragma unroll
      for (int i = 0; i < 31; i++) acc[i] = fma(-cj[i], x, acc[i + 1]);
      acc[31] = 0.0;
      if (lane < m) R[k * rs + lane] = x;  // zero above the diagonal: lanes > k never received a contribution
    }
  }
  asm volatile("bar.sync %0, 64;" ::"r"(bar) : "memory");  // R holds L^-1 for both warps
  return ok;
}
}  // namespace

// MODE 0: reference level, 1: non-reference level, 2: prediction blocks (outG = Hpred receives H, outRi = sd),
// 3: forward-only prediction (new rows of Model::predict_new): the panel carries w_pa in one extra column, and the forward
// sweep alone gives mean = Z'v = K_{u,pa} K_pa^-1 w_pa (into predG) and sd = sqrt(K_uu - diag(Z'Z)) (into predRi), both
// indexed by rioff; no backward sweep, no H.
// phase (MODE 1, childless blocks only): 0 = everything; 1 = forward half: Z, the diagonal Schur complements and the
// log-density pieces, with Z parked in G's storage (nobody reads a childless block's G unless its slot becomes the
// current one); 2 = the deferred half: Z is read back, scaled and pushed through the backward sweep into G.
// In phases 1 and 2 the panel has one extra column that carries w_pa, so that v = L^-1 w_pa and with it
// H w_pa = Z'v come out of the forward sweep.
template <int MODE>
__device__ __forceinline__ void
build_level_body(const DevTree& T, const DevSlots& D, int rel, double* __restrict__ predG, double* __restrict__ predRi, int want_H,
                 const int* __restrict__ grp_slot0, const int* __restrict__ grp_nn, const double* __restrict__ w,
                 int* __restrict__ fail, int ns, int phase_arg, unsigned long long* __restrict__ prof, const int* __restrict__ run_flag) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // bit 2 of the phase argument: the launch runs while the Gibbs sweep is still rewriting w (st_model.cu: the early levels of a
  // BUILD overlap the sweep on a second stream); its log-density pieces e' prec e are then left to an LLW pass over the
  // finished slot, everything that depends on theta alone (G, Ri, logdet) is written as usual
  const int phase = phase_arg & 3;
  const bool density = (phase_arg & 4) == 0;
  // conditional launches of the device-resident chain (deferred half after an accepted proposal, prediction weights after
  // theta moved): the flag was written by an earlier kernel of the stream and is the same for every thread
  if (run_flag != nullptr && *run_flag == 0) return;
  // which theta-slot: read from the chain state in device memory (accept_make_change flips it there)
  const int phys = D.chain->cur ^ rel;
  const DevSlot S = pick_slot(D, phys);
  double* __restrict__ outG = (MODE >= 2) ? predG : S.G;
  double* __restrict__ outH = (MODE < 2 && want_H) ? S.H : nullptr;
  double* __restrict__ outRi = (MODE >= 2) ? predRi : S.Ri;
  const CovTab& tab = D.chain->tab[phys];
  __shared__ CovTabS ct;
  __shared__ int s_cm[kMaxChain], s_crow[kMaxChain + 1], s_crow0g[kMaxChain], s_cgs[kMaxChain];
  __shared__ long long s_cgoff[kMaxChain];
  __shared__ int s_nm[kMaxGroupNodes], s_nc0[kMaxGroupNodes + 1], s_nrow0[kMaxGroupNodes], s_ngs[kMaxGroupNodes], s_nRb[kMaxGroupNodes];
  __shared__ long long s_ngoff[kMaxGroupNodes], s_nrioff[kMaxGroupNodes], s_nmoff[kMaxGroupNodes];
  __shared__ double s_nlogdet[kMaxGroupNodes];
  __shared__ int s_sumRb, s_maxmd;

  const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nth >> 5;
  const int s0 = grp_slot0[blockIdx.x], nn = grp_nn[blockIdx.x];
  const int k = T.k[s0], P = T.P[s0];

  long long tprev = clock64();
  auto mark = [&](int ph) {
    if (prof && tid == 0) { const long long t = clock64(); atomicAdd(prof + ph, (unsigned long long)(t - tprev)); tprev = t; }
  };
  // Programmatic dependent launch: the next level's CTAs may be scheduled as soon as SMs free up (they fill the tail of
  // this launch and run their setup and covariance panel, which depend on nothing this launch writes) ...
  asm volatile("griddepcontrol.launch_dependents;");
  load_covtab(ct, tab);
  // ---- setup: metadata of the chain and of the group's blocks
  {
    const int coff = T.chain_off[s0];
    for (int j = tid; j < k; j += nth) {
      const int a = T.chain[coff + j];
      s_cm[j] = T.m[a]; s_crow[j] = T.chain_poff[coff + j]; s_crow0g[j] = T.row0[a];
      // limited trees: the (single) parent contributes its MARGINAL factor rows [-chol(K_pp)^-1 | 0] (:901-903)
      s_cgoff[j] = T.limited ? T.moff[a] : T.goff[a];
      s_cgs[j] = T.limited ? ((T.m[a] + 3) & ~3) : T.gs[a];
    }
    for (int d = tid; d < nn; d += nth) {
      s_nm[d] = T.m[s0 + d]; s_nrow0[d] = T.row0[s0 + d]; s_ngoff[d] = T.goff[s0 + d]; s_ngs[d] = T.gs[s0 + d];
      s_nrioff[d] = T.rioff[s0 + d];
      s_nmoff[d] = (MODE == 0 && T.limited) ? T.moff[s0 + d] : -1;
    }
  }
  __syncthreads();
  if (tid == 0) {
    int c = 0, rb = 0, mx = 1;
    for (int d = 0; d < nn; d++) {
      s_nc0[d] = c; s_nRb[d] = rb;
      c += s_nm[d];
      if (MODE == 0) rb += rb_doubles(s_nm[d]);
      mx = max(mx, s_nm[d]);
    }
    s_nc0[nn] = c; s_sumRb = rb; s_maxmd = mx; s_crow[k] = P;  // (limited trees keep a second set of matrices behind the first)
  }
  __syncthreads();
  const int ncols = s_nc0[nn];
  const int xcol = ((MODE == 1 && phase != 0) || MODE == 3) ? 1 : 0;
  const int nmat = (MODE == 0 && T.limited) ? 2 : 1;  // limited trees factorise K_uu (marginal) next to the Schur complement
  const BuildPlan pl = build_plan(P, ncols + xcol, nmat * s_sumRb, s_maxmd, ns, (MODE == 0) ? min(nmat * nn, kBuildMaxThreads / 32) : 0, nwarps);
  const int Ppad = pl.Ppad, NCp = pl.NCp, NT = pl.NT, LD = pl.LD, SA = pl.SA, slotsz = pl.slot;
  double* base = reinterpret_cast<double*>(smem_raw);
  double* panel = base + pl.o_panel;
  double* ring = base + pl.o_ring;
  double* Rb = ring;  // the Schur complements live in the ring while it is idle (between the sweeps)
  double* pxs = base + pl.o_pxs;
  double* pys = base + pl.o_pys;
  double* wpa = base + pl.o_wpa;
  double* cxs = base + pl.o_cxs;
  double* cys = base + pl.o_cys;
  double* wcol = base + pl.o_wcol;
  double* tvec = base + pl.o_tvec;
  double* gw = base + pl.o_gw;
  double* rdiag = base + pl.o_rdiag;
  long long* rowsrc = reinterpret_cast<long long*>(base + pl.o_rowsrc);
  long long* colbase = reinterpret_cast<long long*>(base + pl.o_colbase);
  double* vtmp = base + pl.o_vtmp;
  double* s_cb = base + pl.o_scr;
  int* pq = reinterpret_cast<int*>(base + pl.o_scr + 2 * (size_t)Ppad);
  int* rowlen = reinterpret_cast<int*>(base + pl.o_rowlen);
  int* cq = reinterpret_cast<int*>(base + pl.o_cq);
  int* colnode = reinterpret_cast<int*>(base + pl.o_colnode);

  // ---- phase 1: per parent row (= row of the chain's factor) and per column metadata, one pass (independent loads)
  for (int r = tid; r < Ppad; r += nth) {
    if (r < P) {
      int j = 0;
      while (j + 1 < k && r >= s_crow[j + 1]) j++;
      const int t = r - s_crow[j], g = s_crow0g[j] + t;
      pxs[r] = T.cx[g]; pys[r] = T.cy[g]; pq[r] = T.mvq[g]; wpa[r] = w[g];
      rowsrc[r] = s_cgoff[j] + (long long)t * s_cgs[j];
      rowlen[r] = s_crow[j] + s_cm[j];  // [G_a | -Ri_a]: the entries above Ri's diagonal are stored zeros
    } else {
      pxs[r] = 0; pys[r] = 0; pq[r] = 0; wpa[r] = 0; rowsrc[r] = 0; rowlen[r] = 0;
    }
  }
  for (int c = tid; c < LD; c += nth) {
    tvec[c] = 0; gw[c] = 0; rdiag[c] = 0;
    if (c < ncols) {
      int d = 0;
      while (d + 1 < nn && c >= s_nc0[d + 1]) d++;
      const int t = c - s_nc0[d], g = s_nrow0[d] + t;
      cxs[c] = T.cx[g]; cys[c] = T.cy[g]; cq[c] = T.mvq[g]; colnode[c] = d;
      colbase[c] = s_ngoff[d] + (long long)t * s_ngs[d];
      wcol[c] = (MODE >= 2) ? 0.0 : w[g];
    } else {
      cxs[c] = 0; cys[c] = 0; cq[c] = 0; colnode[c] = -1; colbase[c] = -1; wcol[c] = 0;
    }
  }
  __syncthreads();
  mark(0);

  // ---- phase 2: covariance panel K_{pa,u}; rows >= P and columns past the group's are zero
  const bool completing = (MODE == 1 && phase == 2);
  {
    // zero fill: the columns past the group's (all rows) and the rows past P
    const int npadc = LD - ncols;
    for (int e = tid; e < Ppad * npadc; e += nth) { const int i = e / npadc; panel[(size_t)i * LD + ncols + (e - i * npadc)] = 0.0; }
    for (int e = tid; e < (Ppad - P) * ncols; e += nth) { const int i = e / ncols; panel[(size_t)(P + i) * LD + (e - i * ncols)] = 0.0; }
  }
  if (completing) {
    // deferred half: the panel is Z, parked (unscaled) in G's storage by the forward half.  It goes straight into the
    // panel with 8-byte cp.async (the transposition rules out wider copies) and lands together with the first stage of
    // the sweep; the 1 / sqrt(R_ii) scaling is applied to the sweep's outputs.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    for (int c = tid; c < ncols; c += nth) rdiag[c] = outRi[s_nrioff[colnode[c]] + (c - s_nc0[colnode[c]])];
    for (int e = tid; e < ncols * P; e += nth) {
      const int c = e / P, i = e - c * P;
      asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(panel + (size_t)i * LD + c)),
                   "l"(S.G + colbase[c] + i) : "memory");
    }
  }
  if (!completing) {
    // lanes over columns, warps over rows, kCovIlp independent evaluations in flight per thread.  The last, partial run of
    // 32 columns is packed: with w = the power of two that holds them, a warp covers 32 / w rows at once.
    auto cov_cols = [&](int c, bool act, int ifirst, int istep) {
      const double xc = cxs[c], yc = cys[c];
      const int qc = cq[c];
      int i = ifirst;
      for (; i + (kCovIlp - 1) * istep < P; i += kCovIlp * istep) {
        double v[kCovIlp];
#pragma unroll
        for (int u = 0; u < kCovIlp; u++) v[u] = cov_eval(ct, pxs[i + u * istep], pys[i + u * istep], pq[i + u * istep], xc, yc, qc);
#pragma unroll
        for (int u = 0; u < kCovIlp; u++) if (act) panel[(size_t)(i + u * istep) * LD + c] = v[u];
      }
      for (; i < P; i += istep) {
        const double v = cov_eval(ct, pxs[i], pys[i], pq[i], xc, yc, qc);
        if (act) panel[(size_t)i * LD + c] = v;
      }
    };
    const int cfull = ncols & ~31, nrem = ncols - cfull;
    for (int c = lane; c < cfull; c += 32) cov_cols(c, true, warp, nwarps);
    if (nrem > 0) {
      int wl = 0;
      while ((1 << wl) < nrem) wl++;
      const int cl = lane & ((1 << wl) - 1), rp = 32 >> wl;
      cov_cols(cfull + min(cl, nrem - 1), cl < nrem, warp * rp + (lane >> wl), nwarps * rp);
    }
  }
  if (xcol && !completing) {
    __syncthreads();  // the zero fill above covered the columns past the group's
    for (int i = tid; i < Ppad; i += nth) panel[(size_t)i * LD + ncols] = wpa[i];  // extra column: w_pa (zero past P)
  }
  // (the first __syncthreads of the sweep below publishes the panel)
  mark(1);

  const int nstg = Ppad / RS;
  // warp roles in the sweeps: warp < nfull owns column tile `warp`; the other tiles are shared by two warps that split
  // the reduction range (the FP64 pipe is per SM sub-partition: this evens out the load of the four of them)
  const int npair = pl.npair, nfull = NT - npair;
  const int my_nt = (warp < NT) ? warp : ((warp < NT + npair) ? warp - npair : -1);
  const bool paired = my_nt >= nfull, second = warp >= NT;
  double* red = base + pl.o_scr + (size_t)(paired ? my_nt - nfull : 0) * 128;
  const int bar_id = 1 + (paired ? my_nt - nfull : 0);
  auto pair_sync = [&]() { asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory"); };
  // 16-byte cp.async with zero fill of the bytes past `valid_bytes` (0, 8 or 16)
  auto cp16 = [](double* dst, const double* src, int valid_bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src), "r"(valid_bytes) : "memory");
  };
  // threads per staged row: a power of two, so that the (row, chunk) split of a stage needs no division
  int tpr_log = 0;
  while ((RS << (tpr_log + 1)) <= nth) tpr_log++;
  // stage of the forward sweep: rows [r0, r0 + 16) of the chain's factor, columns [0, r0 + 16)
  auto issue_fwd = [&](int st, double* slot) {
    const int r0 = st * RS, kext = r0 + RS;
    const int rr = tid >> tpr_log;
    if (rr >= RS) return;
    const int r = r0 + rr, len = rowlen[r];
    const double* src = S.G + rowsrc[r];
    double* dst = slot + rr * SA;
    for (int c2 = (tid & ((1 << tpr_log) - 1)) * 2; c2 < kext; c2 += 2 << tpr_log) {
      const int valid = min(max(len - c2, 0), 2);
      cp16(dst + c2, src + (valid ? c2 : 0), 8 * valid);
    }
  };
  // stage of the backward sweep: columns [r0, r0 + 16) of rows [r0, Ppad)
  auto issue_bwd = [&](int st, double* slot) {
    const int r0 = st * RS, c2 = (tid & 7) * 2;
    for (int r = r0 + (tid >> 3); r < Ppad; r += nth >> 3) {
      const int valid = min(max(rowlen[r] - (r0 + c2), 0), 2);
      cp16(slot + (r - r0) * ST + c2, S.G + rowsrc[r] + (valid ? r0 + c2 : 0), 8 * valid);
    }
  };

  // ---- phase 3: Z = L^-1 K in place, bottom rows first (row r of Z needs rows <= r of K)
  // ... and wait here, before the first read of the ancestors' row blocks, until the previous launches have completed
  // and their writes are visible (a no-op for a launch without the programmatic attribute)
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int nfw = completing ? 0 : nstg;
  if (ns == 2 && nfw > 0) issue_fwd(nfw - 1, ring);
  for (int i = 0; i < nfw; i++) {
    const int st = nfw - 1 - i;
    double* slot = ring + ((ns == 2) ? (i & 1) * slotsz : 0);
    if (ns == 1) issue_fwd(st, slot);
    __pipeline_commit();
    __pipeline_wait_prior(0);
    __syncthreads();
    if (ns == 2 && i + 1 < nfw) issue_fwd(st - 1, ring + ((i + 1) & 1) * slotsz);
    if (my_nt >= 0) {
      const int r0 = st * RS;
      const double* ap = slot + (lane >> 2) * SA + (lane & 3);
      const double* bp = panel + (size_t)(lane & 3) * LD + 8 * my_nt + (lane >> 2);
      double c0[2] = {0, 0}, c1[2] = {0, 0}, d0[2] = {0, 0}, d1[2] = {0, 0};
      const int K0 = r0 + 8, K1 = r0 + 16;  // the upper m-tile (rows r0 .. r0+7) has no entries past column r0 + 7
      const int Kmid = ((K1 >> 1) + 7) & ~7;
      const int kbeg = (paired && second) ? Kmid : 0, kend = (paired && !second) ? Kmid : K1;
#pragma unroll 2
      for (int kk = kbeg; kk < kend; kk += 8) {
        const double b0 = bp[(size_t)kk * LD], b1 = bp[(size_t)(kk + 4) * LD];
        const double a1 = ap[8 * SA + kk], a3 = ap[8 * SA + kk + 4];
        dmma(c1, a1, b0); dmma(d1, a3, b1);
        if (kk < K0) {
          const double a0 = ap[kk], a2 = ap[kk + 4];
          dmma(c0, a0, b0); dmma(d0, a2, b1);
        }
      }
      double2 z0 = make_double2(c0[0] + d0[0], c0[1] + d0[1]), z1 = make_double2(c1[0] + d1[0], c1[1] + d1[1]);
      if (paired && second) {
        *reinterpret_cast<double2*>(red + lane * 4) = z0;
        *reinterpret_cast<double2*>(red + lane * 4 + 2) = z1;
        pair_sync();
      } else {
        if (paired) {
          pair_sync();
          const double2 p0 = *reinterpret_cast<const double2*>(red + lane * 4), p1 = *reinterpret_cast<const double2*>(red + lane * 4 + 2);
          z0.x += p0.x; z0.y += p0.y; z1.x += p1.x; z1.y += p1.y;
        }
        // the staged rows are [G | -Ri] = -L^-1
        double* o = panel + (size_t)(r0 + (lane >> 2)) * LD + 8 * my_nt + 2 * (lane & 3);
        *reinterpret_cast<double2*>(o) = make_double2(-z0.x, -z0.y);
        *reinterpret_cast<double2*>(o + (size_t)8 * LD) = make_double2(-z1.x, -z1.y);
      }
    }
    if (ns == 1) __syncthreads();
  }
  __syncthreads();
  mark(2);

  // ---- phase 4/5: Schur complement and its inverse Cholesky factor
  if (MODE == 0) {
    const int sumRb = s_sumRb;
    for (int e = tid; e < nmat * sumRb; e += nth) Rb[e] = 0.0;
    __syncthreads();
    // one 8 x 8 tile of the lower triangle per item; the FP64 pipe is per SM sub-partition, so the items are dealt to a
    // multiple of four warps
    const int nwe = (nwarps >= 4) ? (nwarps & ~3) : nwarps;
    int total = 0;
    for (int d = 0; d < nn; d++) { const int mt = (s_nm[d] + 7) >> 3; total += mt * (mt + 1) / 2; }
    for (int item = warp; item < total && warp < nwe; item += nwe) {
      int d = 0, rem = item;
      for (;; d++) {
        const int mt = (s_nm[d] + 7) >> 3, cnt = mt * (mt + 1) / 2;
        if (rem < cnt) break;
        rem -= cnt;
      }
      int ti = 0;
      while ((ti + 1) * (ti + 2) / 2 <= rem) ti++;
      const int tj = rem - ti * (ti + 1) / 2;
      const int md = s_nm[d], c0d = s_nc0[d], rs = rb_stride(md);
      const double* ap = panel + (size_t)(lane & 3) * LD + min(c0d + 8 * ti + (lane >> 2), LD - 1);
      const double* bp = panel + (size_t)(lane & 3) * LD + min(c0d + 8 * tj + (lane >> 2), LD - 1);
      double c0[2] = {0, 0}, d0[2] = {0, 0}, c1[2] = {0, 0}, d1[2] = {0, 0};
#pragma unroll 2
      for (int kk = 0; kk < Ppad; kk += 16) {
        dmma(c0, ap[(size_t)kk * LD], bp[(size_t)kk * LD]);
        dmma(d0, ap[(size_t)(kk + 4) * LD], bp[(size_t)(kk + 4) * LD]);
        dmma(c1, ap[(size_t)(kk + 8) * LD], bp[(size_t)(kk + 8) * LD]);
        dmma(d1, ap[(size_t)(kk + 12) * LD], bp[(size_t)(kk + 12) * LD]);
      }
      const int i = 8 * ti + (lane >> 2), j = 8 * tj + 2 * (lane & 3);
      double* R = Rb + s_nRb[d];
#pragma unroll
      for (int e = 0; e < 2; e++)
        if (i < md && j + e <= i) {
          const double kuu = cov_eval(ct, cxs[c0d + i], cys[c0d + i], cq[c0d + i], cxs[c0d + j + e], cys[c0d + j + e], cq[c0d + j + e]);
          R[i * rs + j + e] = kuu - ((c0[e] + d0[e]) + (c1[e] + d1[e]));
          if (nmat == 2) R[sumRb + i * rs + j + e] = kuu;  // K_uu itself: its factor is what the children stream
        }
    }
    __syncthreads();
    mark(3);
    // one warp pair per matrix (warps 2i and 2i+1 sit on different SM sub-partitions); named barriers 1.. are free here,
    // the sweeps that use them are over
    for (int x = warp >> 1; x < nmat * nn; x += nwarps >> 1) {
      const int d = x % nn, which = x / nn;  // which = 1: the marginal K_uu of a limited tree
      const int md = s_nm[d], rs = rb_stride(md), role = warp & 1;
      double* R = Rb + which * sumRb + s_nRb[d];
      bool okc = true;
      long long tc0 = 0;
      if (prof && tid == 0) tc0 = clock64();
      if (md <= 32) {
        double* scr = s_cb + (warp >> 1) * 160;
        okc = pair_chol_inv32(R, md, rs, scr, scr + 128, lane, role, 1 + (warp >> 1));
        if (prof && tid == 0) atomicAdd(prof + 8, (unsigned long long)(clock64() - tc0));
      } else if (role == 0) {
        okc = warp_chol(R, md, rs, lane);
        if (okc) warp_inv_lower_inplace(R, md, rs, vtmp + (warp >> 1) * (s_maxmd + 2), lane);
      }
      if (role == 0) {
        if (!okc) {
          if (lane == 0) atomicAdd(fail, 1);
          __syncwarp();
          for (int e = lane; e < md * rs; e += 32) R[e] = 0.0;
        }
        if (lane == 0 && which == 0) s_nlogdet[d] = okc ? 0.0 : -1.0;  // flag, replaced by the log-determinant below
      }
    }
    __syncthreads();
    mark(4);
    // Ri to global memory: the stand-alone tile (Gibbs, LLW) and the [G | -Ri] row block (children's BUILD)
    for (int d = 0; d < nn; d++) {
      const int md = s_nm[d], rs = rb_stride(md), trs = tile_rs(md), gsd = s_ngs[d];
      const double* R = Rb + s_nRb[d];
      double* ori = outRi + s_nrioff[d];
      double* og = outG + s_ngoff[d] + P;
      for (int e = tid; e < md * trs; e += nth) {
        const int r = e / trs, c = e - r * trs;
        const double v = (c < md) ? R[r * rs + c] : 0.0;
        ori[e] = v;
        if (c < md) og[(size_t)r * gsd + c] = -v;
      }
    }
    if (nmat == 2)  // limited trees: the marginal factor rows [-chol(K_uu)^-1 | 0] for the children's BUILD
      for (int d = 0; d < nn; d++) {
        if (s_nmoff[d] < 0) continue;
        const int md = s_nm[d], rs = rb_stride(md), ms = (md + 3) & ~3;
        const double* M2 = Rb + sumRb + s_nRb[d];
        double* om = outG + s_nmoff[d];
        for (int e = tid; e < md * md; e += nth) { const int r = e / md, c = e - r * md; om[(size_t)r * ms + c] = -M2[r * rs + c]; }
      }
    // t = Ri w_u (:912-913 via e = w_u - H w_pa: Ri e = Ri w_u - G w_pa) and logdet = sum log diag(Ri) (:966)
    for (int c = tid; c < ncols; c += nth) {
      const int d = colnode[c], c0d = s_nc0[d], r = c - c0d;
      const double* Rr = Rb + s_nRb[d] + r * rb_stride(s_nm[d]);
      double t0 = 0, t1 = 0;
      int c2 = 0;
      for (; c2 + 1 <= r; c2 += 2) { t0 = fma(Rr[c2], wcol[c0d + c2], t0); t1 = fma(Rr[c2 + 1], wcol[c0d + c2 + 1], t1); }
      if (c2 <= r) t0 = fma(Rr[c2], wcol[c0d + c2], t0);
      tvec[c] = t0 + t1;
    }
    __syncthreads();
    for (int d = warp; d < nn; d += nwarps) {
      const int md = s_nm[d], rs = rb_stride(md);
      const double* R = Rb + s_nRb[d];
      const bool okc = s_nlogdet[d] == 0.0;
      double ld = 0;
      for (int r = lane; r < md; r += 32) ld += okc ? log(R[r * rs + r]) : 0.0;
      ld = warp_sum(ld);
      __syncwarp();
      if (lane == 0) s_nlogdet[d] = ld;
    }
    __syncthreads();
  } else if (!completing) {
    // diag(Z'Z) and Z'v per column: the rows are split into parts of 32 so that every thread has work (a narrow group has
    // far fewer columns than the CTA has threads); partial sums in the idle ring, summed in a fixed order that depends
    // on P alone (the eager and the deferred scheme, whose panels differ by the w_pa column, stay bit-identical)
    const int rpp = 32, np = (Ppad + rpp - 1) / rpp;  // np * 2 * NCp <= Ppad * NCp / 8 doubles: inside one backward stage
    double* part = ring;
    for (int item = tid; item < np * NCp; item += nth) {
      const int pt = item / NCp, c = item - pt * NCp;
      const int pend = min(Ppad, (pt + 1) * rpp);
      double q0 = 0, q1 = 0, q2 = 0, q3 = 0, g0 = 0, g1 = 0;
      for (int pp = pt * rpp; pp < pend; pp += 4) {
        const double z0 = panel[(size_t)pp * LD + c], z1 = panel[(size_t)(pp + 1) * LD + c];
        const double z2 = panel[(size_t)(pp + 2) * LD + c], z3 = panel[(size_t)(pp + 3) * LD + c];
        q0 = fma(z0, z0, q0); q1 = fma(z1, z1, q1); q2 = fma(z2, z2, q2); q3 = fma(z3, z3, q3);
        if (xcol) {  // H w_pa = Z'v with v = L^-1 w_pa in the extra column
          const double* v = panel + (size_t)pp * LD + ncols;
          g0 = fma(z0, v[0], g0); g1 = fma(z1, v[LD], g1); g0 = fma(z2, v[2 * LD], g0); g1 = fma(z3, v[3 * LD], g1);
        }
      }
      part[(size_t)(2 * pt) * NCp + c] = (q0 + q1) + (q2 + q3);
      part[(size_t)(2 * pt + 1) * NCp + c] = g0 + g1;
    }
    __syncthreads();
    for (int c = tid; c < NCp; c += nth) {
      const int d = (c < ncols) ? colnode[c] : -1;
      if (d < 0) continue;
      double qs = 0, gsum = 0;
      for (int pt = 0; pt < np; pt++) { qs += part[(size_t)(2 * pt) * NCp + c]; gsum += part[(size_t)(2 * pt + 1) * NCp + c]; }
      const double R = cov_eval(ct, cxs[c], cys[c], cq[c], cxs[c], cys[c], cq[c]) - qs;
      const bool ok = (R > 0.0) && isfinite(R);
      const int t = c - s_nc0[d];
      if (MODE == 1) {
        if (!ok) atomicAdd(fail, 1);
        const double ri = ok ? 1.0 / sqrt(R) : 0.0;  // ccholprecdiag (:945)
        rdiag[c] = ri;
        outRi[s_nrioff[d] + t] = ri;
        tvec[c] = ri * wcol[c];
        if (xcol) gw[c] = ri * gsum;  // G w_pa
      } else if (MODE == 3) {
        outG[s_nrioff[d] + t] = gsum;
        outRi[s_nrioff[d] + t] = ok ? sqrt(R) : 0.0;  // as in-chain prediction (:1316-1322)
      } else {
        outRi[s_nrioff[d] + t] = ok ? sqrt(R) : 0.0;  // predict_std zeroes the sd when the Cholesky fails (:1316-1322)
      }
    }
    __syncthreads();
    mark(3);
    mark(4);
  }

  // ---- backward sweep: out' = L^-T panel, written straight to global memory (row block layout of the group's blocks)
  // scale: column c of the result is multiplied by rdiag[c] (non-reference rows: G_i = H_i / sqrt(R_ii), :945-948)
  auto bwd_sweep = [&](double* __restrict__ out, bool do_gw, bool scale) {
    double gacc[2] = {0, 0};
    if (ns == 2 && nstg > 0) issue_bwd(0, ring);
    for (int i = 0; i < nstg; i++) {
      double* slot = ring + ((ns == 2) ? (i & 1) * slotsz : 0);
      if (ns == 1) issue_bwd(i, slot);
      __pipeline_commit();
      __pipeline_wait_prior(0);
      __syncthreads();
      if (ns == 2 && i + 1 < nstg) issue_bwd(i + 1, ring + ((i + 1) & 1) * slotsz);
      if (my_nt >= 0) {
        const int r0 = i * RS, nk = Ppad - r0;
        const double* ap = slot + (lane & 3) * ST + (lane >> 2);  // A[m][k] = stage[k][m] (transposed use)
        const double* bp = panel + (size_t)(r0 + (lane & 3)) * LD + 8 * my_nt + (lane >> 2);
        double c0[2] = {0, 0}, c1[2] = {0, 0}, d0[2] = {0, 0}, d1[2] = {0, 0};
        const int Kmid = ((nk >> 1) + 7) & ~7;
        const int kbeg = (paired && second) ? Kmid : 0, kend = (paired && !second) ? Kmid : nk;
#pragma unroll 2
        for (int kk = kbeg; kk < kend; kk += 8) {
          const double b0 = bp[(size_t)kk * LD], b1 = bp[(size_t)(kk + 4) * LD];
          const double a0 = ap[kk * ST], a2 = ap[(kk + 4) * ST];
          dmma(c0, a0, b0); dmma(d0, a2, b1);
          if (kk >= 8) {  // rows r0 .. r0+7 of the stage have no entries in columns r0+8 .. r0+15 (lower-triangular factor)
            const double a1 = ap[kk * ST + 8], a3 = ap[(kk + 4) * ST + 8];
            dmma(c1, a1, b0); dmma(d1, a3, b1);
          }
        }
        double2 z0 = make_double2(c0[0] + d0[0], c0[1] + d0[1]), z1 = make_double2(c1[0] + d1[0], c1[1] + d1[1]);
        if (paired && second) {
          *reinterpret_cast<double2*>(red + lane * 4) = z0;
          *reinterpret_cast<double2*>(red + lane * 4 + 2) = z1;
          pair_sync();
        } else {
          if (paired) {
            pair_sync();
            const double2 p0 = *reinterpret_cast<const double2*>(red + lane * 4), p1 = *reinterpret_cast<const double2*>(red + lane * 4 + 2);
            z0.x += p0.x; z0.y += p0.y; z1.x += p1.x; z1.y += p1.y;
          }
          const int r = r0 + (lane >> 2), c = 8 * my_nt + 2 * (lane & 3);
          const long long cb0 = colbase[c], cb1 = colbase[c + 1];
          const double sc0 = scale ? -rdiag[c] : -1.0, sc1 = scale ? -rdiag[c + 1] : -1.0;
          const double v00 = sc0 * z0.x, v01 = sc1 * z0.y, v10 = sc0 * z1.x, v11 = sc1 * z1.y;
          if (r < P) {
            if (cb0 >= 0) out[cb0 + r] = v00;
            if (cb1 >= 0) out[cb1 + r] = v01;
          }
          if (r + 8 < P) {
            if (cb0 >= 0) out[cb0 + r + 8] = v10;
            if (cb1 >= 0) out[cb1 + r + 8] = v11;
          }
          if (do_gw) {
            const double w0 = wpa[r], w1 = wpa[r + 8];  // zero past P
            gacc[0] = fma(v00, w0, fma(v10, w1, gacc[0]));
            gacc[1] = fma(v01, w0, fma(v11, w1, gacc[1]));
          }
        }
      }
      if (ns == 1) __syncthreads();
    }
    if (do_gw && warp < NT) {  // (warps >= NT are second halves) G w_pa per column: fixed-order reduction over the lanes that share the column
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) {
        gacc[0] += __shfl_xor_sync(0xffffffffu, gacc[0], o);
        gacc[1] += __shfl_xor_sync(0xffffffffu, gacc[1], o);
      }
      if ((lane >> 2) == 0) { gw[8 * my_nt + 2 * lane] = gacc[0]; gw[8 * my_nt + 2 * lane + 1] = gacc[1]; }
    }
    __syncthreads();
  };

  // wcore = e' prec e = |Ri w_u - G w_pa|^2 (:913 / :950) ; logdet = sum log diag(Ri) (:966)
  auto finalize = [&]() {
    for (int d = warp; d < nn; d += nwarps) {
      const int md = s_nm[d], c0d = s_nc0[d];
      double wc = 0, ld = 0;
      for (int r = lane; r < md; r += 32) {
        const double t = tvec[c0d + r] - gw[c0d + r];
        wc = fma(t, t, wc);
        if (MODE == 1) ld += log(rdiag[c0d + r]);
      }
      wc = warp_sum(wc);
      if (MODE == 1) ld = warp_sum(ld); else ld = s_nlogdet[d];
      if (lane == 0) {
        S.logdet[s0 + d] = ld;
        if (density) S.llcomp[s0 + d] = (double)md * kHl2pi - 0.5 * wc;  // :967-968
      }
    }
  };
  if (MODE == 3) {
    // (mean and sd are out)
  } else if (MODE == 2) {
    bwd_sweep(outG, false, false);  // H of the prediction blocks
  } else if (MODE == 1 && phase == 1) {
    // forward half only: park Z (unscaled) where G will go; the backward sweep runs if and when the slot is taken up
    // (a warp moves 4 rows x 8 columns at a time: with LD = 4 mod 8 the 16 reads of a half-warp fall into 16 different
    // banks, and every four lanes fill one 32-byte sector of a column of Z)
    {
      const int ntile = (ncols + 7) >> 3, Ph = ((P + 7) >> 3) << 2;
      for (int item = warp; item < 2 * ntile; item += nwarps) {
        const int c = 8 * (item >> 1) + (lane >> 2);
        if (c >= ncols) continue;
        double* dst = outG + colbase[c];
        const int ibeg = (item & 1) * Ph, iend = (item & 1) ? P : min(P, Ph);
        for (int i = ibeg + (lane & 3); i < iend; i += 4) dst[i] = panel[(size_t)i * LD + c];
      }
    }
    finalize();
  } else if (completing) {
    __syncthreads();
    bwd_sweep(outG, false, true);
  } else {
    if (outH != nullptr) {
      bwd_sweep(outH, false, false);  // H = K_{u,pa} Kxx_inv (:887), kept only on request
      if (MODE == 0) {  // the sweep used the ring: reload Ri
        const int sumRb = s_sumRb;
        for (int e = tid; e < sumRb; e += nth) Rb[e] = 0.0;
        __syncthreads();
        for (int d = 0; d < nn; d++) {
          const int md = s_nm[d], rs = rb_stride(md), trs = tile_rs(md);
          const double* ori = outRi + s_nrioff[d];
          double* R = Rb + s_nRb[d];
          for (int e = tid; e < md * md; e += nth) { const int r = e / md, c = e - r * md; R[r * rs + c] = ori[r * trs + c]; }
        }
        __syncthreads();
      }
    }
    // Y' = Z Ri' in place
    if (MODE == 0) {
      const int npt = Ppad >> 3;
      const int nwe = (nwarps >= 4) ? (nwarps & ~3) : nwarps;
      for (int item = warp; item < npt * nn && warp < nwe; item += nwe) {
        const int d = item / npt, pt = item - d * npt;
        const int md = s_nm[d], c0d = s_nc0[d], rs = rb_stride(md);
        const double* R = Rb + s_nRb[d];
        const double* ap = panel + (size_t)(8 * pt + (lane >> 2)) * LD;
        const int mt = (md + 7) >> 3, Kmax = (md + 3) & ~3;
        // chunks of four column tiles, last chunk first: a chunk reads columns below its end and writes only its own
        for (int it0 = ((mt - 1) >> 2) << 2; it0 >= 0; it0 -= 4) {
          const int nt = min(4, mt - it0);
          const int Kc = min(8 * (it0 + nt), Kmax);
          const double* bp = R + (8 * it0 + (lane >> 2)) * rs + (lane & 3);
          double acc[4][2] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}};
          for (int kk = 0; kk < Kc; kk += 4) {
            const double a = ap[min(c0d + kk + (lane & 3), LD - 1)];
#pragma unroll
            for (int u = 0; u < 4; u++)
              if (u < nt && kk < 8 * (it0 + u) + 8) dmma(acc[u], a, bp[u * 8 * rs + kk]);
          }
#pragma unroll
          for (int u = 0; u < 4; u++) {
            if (u >= nt) continue;
            const int jl = 8 * (it0 + u) + 2 * (lane & 3);
            double* o = panel + (size_t)(8 * pt + (lane >> 2)) * LD + c0d + jl;
            if (jl < md) o[0] = acc[u][0];
            if (jl + 1 < md) o[1] = acc[u][1];
          }
        }
      }
    }
    __syncthreads();
    mark(5);
    // G = Ri H (bottom-left block of Kxx_invchol(u), tree_utils.cpp:205); non-reference rows: the sweep scales its outputs
    bwd_sweep(outG, true, MODE != 0);
    finalize();
  }
  mark(6);
}

// Two entry points over the same body, because the register hint that suits one hurts the other (measured on C4): the
// non-reference / prediction instantiations run 11 % faster when ptxas is told that one CTA per SM is enough (it
// otherwise squeezes them into 64 registers with spills), the reference instantiation's register-resident Cholesky runs
// 30 % slower with that hint.
__global__ void __launch_bounds__(kBuildMaxThreads)
build_level_kernel_ref(DevTree T, DevSlots D, int rel, double* __restrict__ predG, double* __restrict__ predRi, int want_H,
                       const int* __restrict__ grp_slot0, const int* __restrict__ grp_nn, const double* __restrict__ w,
                       int* __restrict__ fail, int ns, int phase, unsigned long long* __restrict__ prof, const int* __restrict__ run_flag) {
  build_level_body<0>(T, D, rel, predG, predRi, want_H, grp_slot0, grp_nn, w, fail, ns, phase, prof, run_flag);
}
template <int MODE>
__global__ void __launch_bounds__(kBuildMaxThreads, 1)
build_level_kernel(DevTree T, DevSlots D, int rel, double* __restrict__ predG, double* __restrict__ predRi, int want_H,
                   const int* __restrict__ grp_slot0, const int* __restrict__ grp_nn, const double* __restrict__ w,
                   int* __restrict__ fail, int ns, int phase, unsigned long long* __restrict__ prof, const int* __restrict__ run_flag) {
  build_level_body<MODE>(T, D, rel, predG, predRi, want_H, grp_slot0, grp_nn, w, fail, ns, phase, prof, run_flag);
}

template <int MODE>
static cudaError_t launch_build_t(const DevTree& T, const DevSlots& D, int rel, double* predG, double* predRi, int want_H,
                                  const int* grp_slot0, const int* grp_nn, int ngrp, const double* w,
                                  int* fail, int ns, int phase, size_t smem, cudaStream_t st, int nthreads, unsigned long long* prof, bool pdl,
                                  const int* run_flag) {
  auto kern = (MODE == 0) ? build_level_kernel_ref : build_level_kernel<MODE == 0 ? 1 : MODE>;
  static SmemOptIn optin;
  {
    cudaError_t e = ensure_dynamic_smem(kern, smem, optin);
    if (e != cudaSuccess) return e;
  }
  if (!pdl) {
    kern<<<ngrp, nthreads, smem, st>>>(T, D, rel, predG, predRi, want_H, grp_slot0, grp_nn, w, fail, ns, phase, prof, run_flag);
    return cudaGetLastError();
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(ngrp);
  cfg.blockDim = dim3(nthreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, T, D, rel, predG, predRi, want_H, grp_slot0, grp_nn, w, fail, ns, phase, prof, run_flag);
}
cudaError_t launch_build(int mode, const DevTree& T, const DevSlots& D, int rel, double* predG, double* predRi, int want_H,
                         const int* grp_slot0, const int* grp_nn, int ngrp, const double* w, int* fail, int ns, int phase, size_t smem,
                         cudaStream_t st, int nthreads, unsigned long long* prof, bool pdl, const int* run_flag) {
  if (ngrp <= 0) return cudaSuccess;
  if (mode == 0) return launch_build_t<0>(T, D, rel, predG, predRi, want_H, grp_slot0, grp_nn, ngrp, w, fail, ns, phase, smem, st, nthreads, prof, pdl, run_flag);
  if (mode == 1) return launch_build_t<1>(T, D, rel, predG, predRi, want_H, grp_slot0, grp_nn, ngrp, w, fail, ns, phase, smem, st, nthreads, prof, pdl, run_flag);
  if (mode == 2) return launch_build_t<2>(T, D, rel, predG, predRi, want_H, grp_slot0, grp_nn, ngrp, w, fail, ns, phase, smem, st, nthreads, prof, pdl, run_flag);
  return launch_build_t<3>(T, D, rel, predG, predRi, want_H, grp_slot0, grp_nn, ngrp, w, fail, ns, phase, smem, st, nthreads, prof, pdl, run_flag);
}

}  // namespace st
