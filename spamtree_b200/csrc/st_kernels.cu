// st_kernels.cu — sm_100a kernels of the SpamTrees hot path.
//
//  build_level_kernel   BUILD of one tree level (get_loglik_comps_w_std, spamtree_model.cpp:834-998): per work group
//                       (a run of sibling blocks, which share their ancestor chain) the cross-covariance panel
//                       K_{pa,u} is built in shared memory, pushed through the chain's inverse Cholesky factor
//                       (Z = L^-1 K), reduced to the Schur complement R = K_uu - Z'Z, factorised, and pulled back
//                       (H' = L^-T Z) — all without leaving shared memory (SURVEY App. F).  Also used for the
//                       prediction blocks (predict_std, :1234-1358).
//  gibbs_level_kernel   Gibbs update of w for one level (gibbs_sample_w_std, :1011-1226) including the messages to
//                       every ancestor, accumulated by pulling from the direct children (deterministic, no atomics);
//                       its ILOO variant also forms each row's integrated log-likelihood (DESIGN.md §5f).
//  gram_level_kernel    theta-only part of the messages (Sigi_children, :1190-1192), refreshed only after theta changes.
//  llw_kernel           log-density at the current theta with the new w (get_loglik_w_std, :781-826).
//  row kernels          beta / tausq sufficient statistics (:1364-1417), X*beta, device normals, predictive draws.
//
// FP64 throughout; B200 has no tcgen05 FP64 kind, the dense contractions are register-tiled DFMA.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>

#include "st_device.cuh"
#include "st_kernels.cuh"

namespace st {

// ------------------------------------------------------------------------------------------------ GIBBS
// One block per tree block (node).  Shared memory: RiS m*m | Sig m*m | wpa P | gwj (k+1)*m | smu m | wn m | rr m
// REF = 1: full m x m conditional (:1037-1089); REF = 0: row-wise scalars (:1091-1155)
// ILOO: also the integrated log-likelihood of every observed row (DESIGN.md §5f), ll[i] = log N(y_i - xb_i; m_i, v_i + tausq_i)
// with N(m_i, v_i) the prior conditional of w_i given the state the block is drawn from.  ll is node-major; yobs holds y
// node-major with NaN at the rows that are not observed, whose slots of ll the kernel leaves alone.
// Its log-density term; v: the prior conditional's variance, tq: tausq_inv of the row.
__device__ __forceinline__ double iloo_term(double resid, double mean, double v, double tq) {
  const double s2 = v + 1.0 / tq, d = resid - mean;
  return -0.5 * (log(6.283185307179586 * s2) + d * d / s2);
}
template <int REF, bool ILOO>
__global__ void __launch_bounds__(kGibbsThreads)
gibbs_level_kernel(DevTree T, DevSlots D, int slot0, double* __restrict__ w, const double* __restrict__ xb,
                   const double* __restrict__ z, const double* __restrict__ tausq_inv, const double* __restrict__ SigS,
                   double* __restrict__ V, double* probe_sig, double* probe_smu, int* __restrict__ fail,
                   double* __restrict__ ll, const double* __restrict__ yobs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // programmatic dependent launch: the next (shallower) level may start early; it waits below before it reads the
  // messages this level writes (everything before that point depends on ancestors only)
  asm volatile("griddepcontrol.launch_dependents;");
  const DevSlot S = pick_slot(D, D.chain->cur);  // param_data
  const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int sd = slot0 + blockIdx.x;
  const int m = T.m[sd], k = T.k[sd], P = T.P[sd], coff = T.chain_off[sd], row0 = T.row0[sd];
  const int rsm = tile_rs(m), gs = T.gs[sd];
  const int msq = REF ? m * rsm : m;
  double* RiS = reinterpret_cast<double*>(smem_raw);
  double* Sig = RiS + msq;
  double* wpa = Sig + (REF ? m * m : m);
  double* gwj = wpa + P;  // k tiles of m, then the total at [k*m, (k+1)*m)
  double* smu = gwj + (size_t)(k + 1) * m;
  double* wn = smu + m;
  double* rr = wn + m;
  const double* G = S.G + T.goff[sd];  // the block's rows of the chain factor, [G | -Ri | 0], one contiguous run
  const double* Rig = S.Ri + T.rioff[sd];
  const int nch = T.child_ptr[sd + 1] - T.child_ptr[sd];
  const int* ch = T.child_idx + T.child_ptr[sd];
  // chain metadata once, in parallel (no dependent global loads inside the loops below)
  __shared__ int c_m[32], c_po[32], c_r0[32];
  __shared__ long long c_voff[16];
  __shared__ double cbuf[128];  // pivot columns of the factorisation (2 x 64, double-buffered)
  if (tid < k) {
    const int a = T.chain[coff + tid];
    c_m[tid] = T.m[a]; c_po[tid] = T.chain_poff[coff + tid]; c_r0[tid] = T.row0[a];
  }
  for (int c = tid; c < min(nch, 16); c += nth) c_voff[c] = T.voff[ch[c]];
  for (int e = tid; e < msq; e += nth) RiS[e] = Rig[e];
  // loads that depend on nothing computed here are issued now, so that their latency hides under the phases below:
  // the children's Gram sum (into Sig), and per row tausq_inv (wn), tausq_inv (y - XB) (smu) and the normal draw (rr)
  if (REF) {
    const long long so0 = T.soff[sd];
    for (int e = tid; e < m * m; e += nth) Sig[e] = (so0 >= 0) ? SigS[so0 + e] : 0.0;
  }
  for (int a = tid; a < m; a += nth) {
    const double tq = tausq_inv[T.mvq[row0 + a]];
    wn[a] = tq;
    smu[a] = tq * (T.y[row0 + a] - xb[row0 + a]);
    rr[a] = z[row0 + a];
  }
  __syncthreads();
  for (int e = tid; e < P; e += nth) {
    int j = 0;
    while (j + 1 < k && e >= c_po[j + 1]) j++;
    wpa[e] = w[c_r0[j] + (e - c_po[j])];
  }
  __syncthreads();
  // gwj[j][r] = G_j(r,:) w_{a_j}   (pieces of H w_pa scaled by Ri; :1063 / :1103); ancestor fastest: a warp reads adjacent row segments
  for (int e = tid; e < k * m; e += nth) {
    const int r = e / k, j = e - r * k;
    const int mj = c_m[j], po = c_po[j];
    const double* g = G + (size_t)r * gs + po;
    const double* wv = wpa + po;
    double s[4] = {0, 0, 0, 0};
    int pp = 0;
    for (; pp + 8 <= mj; pp += 8) {  // eight independent global loads in flight per thread (this is the first touch of G: HBM latency)
      double x[8];
#pragma unroll
      for (int u = 0; u < 8; u++) x[u] = g[pp + u];
#pragma unroll
      for (int u = 0; u < 8; u++) s[u & 3] = fma(x[u], wv[pp + u], s[u & 3]);
    }
    if (pp + 4 <= mj) {
      double x[4];
#pragma unroll
      for (int u = 0; u < 4; u++) x[u] = g[pp + u];
#pragma unroll
      for (int u = 0; u < 4; u++) s[u] = fma(x[u], wv[pp + u], s[u]);
      pp += 4;
    }
    for (; pp < mj; pp++) s[0] = fma(g[pp], wv[pp], s[0]);
    gwj[j * m + r] = (s[0] + s[1]) + (s[2] + s[3]);
  }
  __syncthreads();
  for (int r = tid; r < m; r += nth) {
    double s = 0;
    for (int j = 0; j < k; j++) s += gwj[j * m + r];
    gwj[k * m + r] = s;
  }
  __syncthreads();
  const double* gw = gwj + (size_t)k * m;
  if (REF) {
    // Sigi_tot = prec + sum_children + diag(tausq_inv)  (:1044-1051), prec = Ri'Ri (:912)
    for (int e = tid; e < m * m; e += nth) {
      const int a = e / m, b = e - a * m;
      double s = 0;
      for (int r = max(a, b); r < m; r++) s = fma(RiS[r * rsm + a], RiS[r * rsm + b], s);
      s += Sig[e];  // sum over the children, prefetched above
      if (a == b) s += wn[a];
      Sig[e] = s;
      if (probe_sig) probe_sig[T.rioff[sd] + e] = s;
    }
    // The factorisation depends on theta and tausq only — not on the children's messages — so it runs BEFORE the wait on the
    // previous (deeper) level: with programmatic dependent launch the 25-pivot latency chains of consecutive levels overlap
    // instead of queueing behind each other, and only the two triangular solves remain on the level-to-level chain.
    __syncthreads();
    bool okc = true;
    double myinv = 0.0;  // 1 / L(lane, lane)
    if (warp == 0) {
      if (m <= 32) {
        // lane i keeps row i of Sigi_tot in registers, rotated so that the pivot column is a[0]; L overwrites Sig
        double a[32];
#pragma unroll
        for (int j = 0; j < 32; j++) a[j] = (lane < m && j <= lane) ? Sig[lane * m + j] : 0.0;
        cbuf[32 + lane] = 0.0;
        cbuf[96 + lane] = 0.0;
        __syncwarp();
        for (int j = 0; j < m; j++) {
          double d = __shfl_sync(0xffffffffu, a[0], j);
          if (!(d > 0.0) || !isfinite(d)) { okc = false; d = 1.0; }
          const double inv = rsqrt(d), sd = d * inv;
          const double l = (lane == j) ? sd : ((lane > j) ? a[0] * inv : 0.0);
          if (lane == j) myinv = inv;
          if (lane >= j && lane < m) Sig[lane * m + j] = l;
          // pivot column to every lane through shared memory (tools/microbench/chol_bench.cu: 388 cycles per pivot,
          // against 1422 with a shuffle per column)
          double* cc = cbuf + (j & 1) * 64;
          cc[lane] = l;
          __syncwarp();
          const double* cj = cc + j + 1;
#pragma unroll
          for (int i = 0; i < 31; i++) a[i] = fma(-l, cj[i], a[i + 1]);
          a[31] = 0.0;
        }
        __syncwarp();
      } else {
        okc = warp_chol(Sig, m, m, lane);
      }
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");  // the children's messages (V) are read from here on
    // Smu_tot = (H'prec)' w_pa + sum_children + tausq_inv (y - XB)  (:1062-1077)
    for (int a = tid; a < m; a += nth) {
      double s = 0;
      for (int r = a; r < m; r++) s = fma(RiS[r * rsm + a], gw[r], s);
      // a child's vector holds its messages by ancestor column; this block's own columns start at P there (its parent set
      // is this block's chain plus this block) — or at 0 in a limited tree, where the parent set is this block alone
      for (int c = 0; c < nch; c++) s += V[(c < 16 ? c_voff[c] : T.voff[ch[c]]) + (T.limited ? 0 : P) + a];
      s += smu[a];  // tausq_inv (y - XB), prefetched above
      smu[a] = s;
      if (probe_smu) probe_smu[row0 + a] = s;
    }
    __syncthreads();
    if (warp == 0) {
      // w = Sc'(Sc Smu + z), Sc = chol(Sigi_tot)^-1 (:1054, :1086), done as two triangular solves
      if (okc && m <= 32) {
        double b = (lane < m) ? smu[lane] : 0.0;
        for (int j = 0; j < m; j++) {  // forward: L x = Smu
          const double xj = __shfl_sync(0xffffffffu, b * myinv, j);
          if (lane == j) b = xj; else if (lane > j && lane < m) b = fma(-Sig[lane * m + j], xj, b);
        }
        double y = (lane < m) ? b + rr[lane] : 0.0;  // z, prefetched above
        for (int j = m - 1; j >= 0; j--) {  // backward: L' w = x + z
          const double wj = __shfl_sync(0xffffffffu, y * myinv, j);
          if (lane == j) y = wj; else if (lane < j) y = fma(-Sig[j * m + lane], wj, y);
        }
        if (lane < m) { wn[lane] = y; w[row0 + lane] = y; }
      } else if (okc) {
        for (int c = 0; c < m; c++) {  // forward: L x = smu
          __syncwarp();
          const double xc = smu[c] / Sig[c * m + c];
          __syncwarp();
          if (lane == 0) smu[c] = xc;
          for (int r = c + 1 + lane; r < m; r += 32) smu[r] -= Sig[r * m + c] * xc;
        }
        __syncwarp();
        for (int r = lane; r < m; r += 32) smu[r] += rr[r];
        for (int c = m - 1; c >= 0; c--) {  // backward: L' w = x
          __syncwarp();
          const double xc = smu[c] / Sig[c * m + c];
          __syncwarp();
          if (lane == 0) smu[c] = xc;
          for (int r = lane; r < c; r += 32) smu[r] -= Sig[c * m + r] * xc;
        }
        __syncwarp();
        for (int r = lane; r < m; r += 32) { wn[r] = smu[r]; w[row0 + r] = smu[r]; }
      }
      if (!okc) {
        if (lane == 0) atomicAdd(fail, 1);
        for (int r = lane; r < m; r += 32) wn[r] = w[row0 + r];
      }
    }
    __syncthreads();
    if (ILOO) {
      // w = L^-T (L^-1 Smu + z), so Sigi_tot w - Smu = L z exactly.  Without row a's own observation the precision is
      // Q'_aa = (Ri'Ri)_aa + (children's Gram)_aa (formed directly, not as Sigi_tot_aa - tausq_inv: no cancellation at small
      // tausq) and the prior conditional of w_a given everything else is N(w_a - [(L z)_a + tausq_inv (resid_a - w_a)] / Q'_aa,
      // 1 / Q'_aa).  rr still holds z here; the loop below overwrites it.
      // Thread a walks row a of L: at step t the threads read a stride of m doubles apart (odd m) or, walking back from the
      // diagonal, m + 1 (even m), so that the stride is odd and the shared-memory reads are free of bank conflicts.  The
      // column of Ri is read at a stride of rsm + 1, odd as well (tile_rs).
      const long long so0 = T.soff[sd];
      const bool back = (m & 1) == 0;
      for (int a = tid; a < m; a += nth) {
        const int i = row0 + a;
        const double yi = yobs[i];
        if (isnan(yi)) continue;  // not observed
        double lz = 0.0, qa = 0.0;
        for (int t = 0; t <= a; t++) {
          const int j = back ? a - t : t;
          lz = fma(Sig[a * m + j], rr[j], lz);
        }
        for (int r = a; r < m; r++) qa = fma(RiS[r * rsm + a], RiS[r * rsm + a], qa);
        if (so0 >= 0) qa += SigS[so0 + (long long)a * m + a];
        const double tq = tausq_inv[T.mvq[i]], res = yi - xb[i], wa = wn[a];
        ll[i] = iloo_term(res, wa - (lz + tq * (res - wa)) / qa, 1.0 / qa, tq);
      }
      __syncthreads();
    }
    for (int r = tid; r < m; r += nth) {
      double s = -gw[r];
      for (int r2 = 0; r2 <= r; r2++) s = fma(RiS[r * rsm + r2], wn[r2], s);
      rr[r] = s;
    }
  } else {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    for (int a = tid; a < m; a += nth) {
      const double ri = RiS[a], prec = ri * ri;
      const double sig = prec + wn[a];                                            // :1123 (tausq_inv prefetched into wn)
      const double sm = ri * gw[a] + smu[a];                                      // :1125-1127
      if (probe_sig) probe_sig[T.rioff[sd] + a] = sig;
      if (probe_smu) probe_smu[row0 + a] = sm;
      double wa;
      if (sig > 0.0 && isfinite(sig)) {
        const double sc = 1.0 / sqrt(sig);
        wa = sc * sc * sm + sc * rr[a];                                           // :1139-1140 (z prefetched into rr)
        w[row0 + a] = wa;
      } else {
        atomicAdd(fail, 1);
        wa = w[row0 + a];
      }
      rr[a] = ri * wa - gw[a];
      // the prior conditional of w_a is N(gw_a / ri, 1 / ri^2): it does not involve w_a.  (ri^2 is formed apart from prec:
      // a second use of prec would keep the compiler from fusing it into sig, and w would change in the last bits.)
      if (ILOO && !isnan(yobs[row0 + a]))
        ll[row0 + a] = iloo_term(yobs[row0 + a] - xb[row0 + a], gw[a] / ri, 1.0 / __dmul_rn(ri, ri), wn[a]);
    }
  }
  __syncthreads();
  // messages to every ancestor (:1158-1207): V_d[J_j] = G_j'(rr + G_j w_{a_j}) + sum over direct children of theirs
  for (int e = tid; e < k * m; e += nth) gwj[e] += rr[e % m];
  __syncthreads();
  double* Vd = V + T.voff[sd];
  // all (ancestor, column) pairs at once: P independent dot products over the block's rows
  for (int e = tid; e < P; e += nth) {
    int j = 0;
    while (j + 1 < k && e >= c_po[j + 1]) j++;
    const int rsj = gs;
    const double* g = G + e;
    const double* vj = gwj + (size_t)j * m;
    double sa[4] = {0, 0, 0, 0};
    int r = 0;
    for (; r + 8 <= m; r += 8) {  // eight independent loads in flight per thread
      double x[8];
#pragma unroll
      for (int u = 0; u < 8; u++) x[u] = g[(size_t)(r + u) * rsj];
#pragma unroll
      for (int u = 0; u < 8; u++) sa[u & 3] = fma(x[u], vj[r + u], sa[u & 3]);
    }
    if (r + 4 <= m) {
      double x[4];
#pragma unroll
      for (int u = 0; u < 4; u++) x[u] = g[(size_t)(r + u) * rsj];
#pragma unroll
      for (int u = 0; u < 4; u++) sa[u] = fma(x[u], vj[r + u], sa[u]);
      r += 4;
    }
    for (; r < m; r++) sa[0] = fma(g[(size_t)r * rsj], vj[r], sa[0]);
    double s = (sa[0] + sa[1]) + (sa[2] + sa[3]);
    if (!T.limited)  // (limited trees: the children's messages stop at this block)
      for (int c = 0; c < nch; c++) s += V[(c < 16 ? c_voff[c] : T.voff[ch[c]]) + e];
    Vd[e] = s;
  }
}

cudaError_t launch_gibbs(int is_ref, const DevTree& T, const DevSlots& D, int slot0, int nslots, double* w,
                         const double* xb, const double* z, const double* tausq_inv, const double* SigS, double* V,
                         double* probe_sig, double* probe_smu, int* fail, size_t smem, cudaStream_t st, bool pdl, double* ll,
                         const double* yobs) {
  if (nslots <= 0) return cudaSuccess;
  static SmemOptIn optin[4];
  const bool iloo = ll != nullptr;
  auto kern = is_ref ? (iloo ? gibbs_level_kernel<1, true> : gibbs_level_kernel<1, false>)
                     : (iloo ? gibbs_level_kernel<0, true> : gibbs_level_kernel<0, false>);
  {
    cudaError_t e = ensure_dynamic_smem(kern, smem, optin[(is_ref ? 1 : 0) + (iloo ? 2 : 0)]);
    if (e != cudaSuccess) return e;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(nslots);
  cfg.blockDim = dim3(kGibbsThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, T, D, slot0, w, xb, z, tausq_inv, SigS, V, probe_sig, probe_smu, fail, ll, yobs);
}

// ------------------------------------------------------------------------------------------------ message Grams
// U_d[j] = G_j'G_j + sum_children U_c[j]  (= sum over the subtree of AK_uP_u_all[J_j, J_j], :1190-1192) and
// SigS_d = sum_children U_c[tile of d]  (= arma::sum(Sigi_children(d), 2), :1049).  One CTA per node.
// Childless children ("fused": the bulk of the tree) never store their own tiles: the parent forms their G_c'G_c
// from their row blocks directly.  The rows (own + fused children) are staged in shared memory in chunks and every
// thread accumulates one 5 x 5 sub-block of the lower triangle of one tile in registers.
__global__ void __launch_bounds__(kGramThreads)
gram_level_kernel(DevTree T, DevSlots D, int slot0, double* __restrict__ U, double* __restrict__ SigS, int rch, int ldx,
                  int stage_off, const int* __restrict__ run_flag) {
  extern __shared__ __align__(16) double gram_smem[];
  // programmatic dependent launch: the next (shallower) level stages its rows and forms its own G'G while this one runs;
  // it waits below, right before it adds the tiles this level stores
  asm volatile("griddepcontrol.launch_dependents;");
  if (run_flag != nullptr && *run_flag == 0) return;  // device-resident chain: only after an accepted proposal
  const DevSlot S = pick_slot(D, D.chain->cur);       // param_data
  __shared__ int t_po[kMaxChain + 1], t_m[kMaxChain + 1], t_item0[kMaxChain + 2], t_uo[kMaxChain + 1], t_to[kMaxChain + 2];
  __shared__ int s_rows;
  __shared__ long long s_rowoff[kGramMaxRows];  // per staged row: offset of the row in S.G and its valid columns
  __shared__ int s_rowncol[kGramMaxRows];
  __shared__ long long s_cu[kGramChildTab];     // per (child, tile): offset of the child's stored tile, -1 when the child is fused
  __shared__ int f_m[kGramFusedTab], f_gs[kGramFusedTab], f_r0[kGramFusedTab + 1];  // fused children: rows, row stride, first staged row
  __shared__ long long f_goff[kGramFusedTab];
  const int tid = threadIdx.x, nth = blockDim.x;
  const int sd = slot0 + blockIdx.x;
  if (T.ufused[sd]) return;
  double* tiles = gram_smem;                 // the assembled tiles (both triangles), tile j at t_to[j]
  double* stage = gram_smem + stage_off;      // rch staged rows of ldx doubles; stage_off = 0: they share the tiles' storage
  const int m = T.m[sd], k = T.k[sd], P = T.P[sd], coff = T.chain_off[sd];
  const int nch = T.child_ptr[sd + 1] - T.child_ptr[sd];
  const int* ch = T.child_idx + T.child_ptr[sd];
  const long long so = T.soff[sd];
  const int ntile = k + (so >= 0 ? 1 : 0);  // the block's own tile exists only through its children
  if (tid <= k) {
    t_po[tid] = (tid < k) ? T.chain_poff[coff + tid] : (T.limited ? 0 : P);  // where the children's rows hold this block's columns
    t_m[tid] = (tid < k) ? T.m[T.chain[coff + tid]] : m;
    t_uo[tid] = (tid < k) ? T.chain_uoff[coff + tid] : 0;
  }
  // the fused children's row blocks, tabulated once (one thread per child: independent loads)
  const bool ftab = nch <= kGramFusedTab;
  if (ftab && tid < nch) {
    const int cc = ch[tid];
    f_m[tid] = T.ufused[cc] ? T.m[cc] : 0;
    f_goff[tid] = T.goff[cc];
    f_gs[tid] = T.gs[cc];
  }
  __syncthreads();
  if (tid == 0) {
    int it = 0, to = 0;
    for (int j = 0; j < ntile; j++) {
      t_item0[j] = it; t_to[j] = to;
      const int nb = (t_m[j] + 4) / 5;
      it += nb * (nb + 1) / 2;
      to += t_m[j] * t_m[j];
    }
    t_item0[ntile] = it; t_to[ntile] = to;
    int rows = m;
    for (int c = 0; c < nch; c++) {
      if (ftab) { f_r0[c] = rows; rows += f_m[c]; }
      else if (T.ufused[ch[c]]) rows += T.m[ch[c]];
    }
    if (ftab) f_r0[nch] = rows;
    s_rows = rows;
  }
  const bool ctab = nch * ntile <= kGramChildTab;
  if (ctab)
    for (int e = tid; e < nch * ntile; e += nth) {
      const int c = e / ntile, jj = e - c * ntile, cc = ch[c];
      // (limited trees: a child carries one tile, this block's; nothing is passed through to the ancestors)
      s_cu[e] = (T.ufused[cc] || (T.limited && jj < k)) ? -1 : T.uoff[cc] + T.chain_uoff[T.chain_off[cc] + (T.limited ? 0 : jj)];
    }
  __syncthreads();
  const int nitems = t_item0[ntile], nrows = s_rows;
  double* Ud = U + T.uoff[sd];
  for (int item0 = 0; item0 < nitems; item0 += nth) {  // (one round unless the chain is very long)
    const int item = item0 + tid;
    const bool act = item < nitems;
    int j = 0, bi = 0, bj = 0;
    if (act) {
      while (item >= t_item0[j + 1]) j++;
      const int rem = item - t_item0[j];
      while ((bi + 1) * (bi + 2) / 2 <= rem) bi++;
      bj = rem - bi * (bi + 1) / 2;
    }
    const int mj = act ? t_m[j] : 1, po = act ? t_po[j] : 0;
    int ca[5], cb[5];
#pragma unroll
    for (int t = 0; t < 5; t++) { ca[t] = po + min(5 * bi + t, mj - 1); cb[t] = po + min(5 * bj + t, mj - 1); }
    double acc[5][5];
#pragma unroll
    for (int x = 0; x < 5; x++)
#pragma unroll
      for (int y = 0; y < 5; y++) acc[x][y] = 0.0;
    // stream the rows through shared memory: row ids 0..m-1 are the block's own (tiles j < k only), then the fused children's
    for (int rbase = 0; rbase < nrows; rbase += rch) {
      const int nr = min(rch, nrows - rbase);
      __syncthreads();
      for (int rr = tid; rr < nr; rr += nth) {  // where does staged row rr live?
        int r = rbase + rr;
        if (r < m) { s_rowoff[rr] = T.goff[sd] + (long long)r * T.gs[sd]; s_rowncol[rr] = P; }
        else if (ftab) {
          int c = 0;
          while (r >= f_r0[c + 1]) c++;  // (children that keep their own tiles have no rows here)
          s_rowoff[rr] = f_goff[c] + (long long)(r - f_r0[c]) * f_gs[c];
          s_rowncol[rr] = T.limited ? m : P + m;
        } else {
          r -= m;
          for (int c = 0; c < nch; c++) {
            const int cc = ch[c];
            if (!T.ufused[cc]) continue;
            const int mc = T.m[cc];
            if (r < mc) { s_rowoff[rr] = T.goff[cc] + (long long)r * T.gs[cc]; s_rowncol[rr] = T.limited ? m : P + m; break; }
            r -= mc;
          }
        }
      }
      __syncthreads();
      {
        const int hl = ldx >> 1;  // 16-byte chunks per staged row; columns past the row's end are zero-filled
        for (int idx = tid; idx < nr * hl; idx += nth) {
          const int rr = idx / hl, x = (idx - rr * hl) * 2;
          const int valid = min(max(s_rowncol[rr] - x, 0), 2);
          asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"((unsigned)__cvta_generic_to_shared(stage + (size_t)rr * ldx + x)),
                       "l"(S.G + s_rowoff[rr] + (valid ? x : 0)), "r"(8 * valid) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
      }
      __syncthreads();
      if (act) {
        const int rb = (j == k) ? max(0, m - rbase) : 0;  // the block's own rows carry no entries of its own tile
        const int re = (T.limited && j < k) ? min(nr, max(0, m - rbase)) : nr;  // limited: the children's rows carry no ancestor tiles
        for (int rr = rb; rr < re; rr++) {
          const double* x = stage + (size_t)rr * ldx;
          double av[5], bv[5];
#pragma unroll
          for (int t = 0; t < 5; t++) { av[t] = x[ca[t]]; bv[t] = x[cb[t]]; }
#pragma unroll
          for (int xx = 0; xx < 5; xx++)
#pragma unroll
            for (int yy = 0; yy < 5; yy++) acc[xx][yy] = fma(av[xx], bv[yy], acc[xx][yy]);
        }
      }
    }
    __syncthreads();  // (the tiles may take the place of the staged rows)
    if (act) {  // both triangles of the tile
      double* tj = tiles + t_to[j];
#pragma unroll
      for (int xx = 0; xx < 5; xx++)
#pragma unroll
        for (int yy = 0; yy < 5; yy++) {
          const int a = 5 * bi + xx, b = 5 * bj + yy;
          if (a < mj && b < mj) { tj[a * mj + b] = acc[xx][yy]; tj[b * mj + a] = acc[xx][yy]; }
        }
    }
  }
  __syncthreads();
  asm volatile("griddepcontrol.wait;" ::: "memory");
  // add the stored tiles of the children that keep theirs, write out (coalesced)
  for (int eg = tid; eg < t_to[ntile]; eg += nth) {
    int j = 0;
    while (eg >= t_to[j + 1]) j++;
    const int e = eg - t_to[j];
    double v = tiles[eg];
    if (ctab) {
      for (int c = 0; c < nch; c++) {
        const long long cu = s_cu[c * ntile + j];
        if (cu >= 0) v += U[cu + e];
      }
    } else {
      for (int c = 0; c < nch; c++) {
        const int cc = ch[c];
        if (!T.ufused[cc] && !(T.limited && j < k)) v += U[T.uoff[cc] + T.chain_uoff[T.chain_off[cc] + (T.limited ? 0 : j)] + e];
      }
    }
    if (j < k) Ud[t_uo[j] + e] = v; else SigS[so + e] = v;
  }
}
cudaError_t launch_gram(const DevTree& T, const DevSlots& D, int slot0, int nslots, double* U, double* SigS, int rch,
                        int ldx, int tile_doubles, int stage_off, int threads, cudaStream_t st, const int* run_flag, bool pdl) {
  if (nslots <= 0) return cudaSuccess;
  const size_t smem = std::max((size_t)tile_doubles, (size_t)stage_off + (size_t)rch * ldx) * sizeof(double);
  static SmemOptIn optin;
  {
    cudaError_t e = ensure_dynamic_smem(gram_level_kernel, smem, optin);
    if (e != cudaSuccess) return e;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(nslots);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, gram_level_kernel, T, D, slot0, U, SigS, rch, ldx, stage_off, run_flag);
}

// ------------------------------------------------------------------------------------------------ LLW
// llcomp[s] = m*hl2pi - 0.5*|Ri w_u - G w_pa|^2  (get_loglik_w_std, :791-813); one warp per node.
// A reference block's rows of the chain factor are [G | -Ri | 0], so its contribution is one streaming product
// |[G | -Ri] [w_pa ; w_u]|^2 over contiguous rows; the warp stages [w_pa ; w_u] in shared memory once.
__global__ void __launch_bounds__(kLlwThreads)
llw_kernel(DevTree T, DevSlots D, int rel, int slot0, int nslots, const double* __restrict__ w, int maxlen,
           double* __restrict__ vrow, int parked) {
  extern __shared__ __align__(16) double llw_smem[];
  const DevSlot S = pick_slot(D, D.chain->cur ^ rel);
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int sd = slot0 + blockIdx.x * (blockDim.x >> 5) + wib;
  if (sd >= slot0 + nslots) return;
  double* wx = llw_smem + (size_t)wib * maxlen;
  const int m = T.m[sd], k = T.k[sd], P = T.P[sd], coff = T.chain_off[sd], row0 = T.row0[sd], gs = T.gs[sd];
  const bool ref = T.isref[sd] != 0;
  const double* G = S.G + T.goff[sd];
  // lane j keeps the metadata of ancestor j (k <= 32)
  int a_m = 0, a_po = 0, a_r0 = 0;
  if (lane < k) {
    const int a = T.chain[coff + lane];
    a_m = T.m[a];
    a_po = T.chain_poff[coff + lane];
    a_r0 = T.row0[a];
  }
  for (int j = 0; j < k; j++) {
    const int mj = __shfl_sync(0xffffffffu, a_m, j), po = __shfl_sync(0xffffffffu, a_po, j), ar0 = __shfl_sync(0xffffffffu, a_r0, j);
    // (parked blocks: the vector is v = L^-1 w_pa, read off the rows of the ancestors: their s = -v, see below)
    for (int t = lane; t < mj; t += 32) wx[po + t] = parked ? -vrow[ar0 + t] : w[ar0 + t];
  }
  const int len = ref ? P + m : P;
  if (ref)
    for (int t = lane; t < m; t += 32) wx[P + t] = w[row0 + t];
  __syncwarp();
  double wc = 0;
  int r = 0;
  for (; r + 1 < m; r += 2) {  // two rows at a time: independent load streams
    const double* g0 = G + (size_t)r * gs;
    const double* g1 = g0 + gs;
    double s0 = 0, s1 = 0;
    for (int c = lane; c < len; c += 32) {
      const double x = wx[c];
      s0 = fma(__ldg(g0 + c), x, s0);
      s1 = fma(__ldg(g1 + c), x, s1);
    }
    s0 = warp_sum(s0);
    s1 = warp_sum(s1);
    if (!ref) {
      const double* Ri = S.Ri + T.rioff[sd];
      if (parked) {  // the row holds Z_r (unscaled): H_r w_pa = Z_r'v, e_r = w_r - H_r w_pa, prec_r = Ri_r^2
        s0 = Ri[r] * (s0 - w[row0 + r]);
        s1 = Ri[r + 1] * (s1 - w[row0 + r + 1]);
      } else {
        s0 -= Ri[r] * w[row0 + r];
        s1 -= Ri[r + 1] * w[row0 + r + 1];
      }
    } else if (vrow != nullptr && lane == 0) {
      vrow[row0 + r] = s0;  // = -(L^-1 [w_pa ; w_u])_r: what the blocks below read as their v
      vrow[row0 + r + 1] = s1;
    }
    wc = fma(s0, s0, wc);
    wc = fma(s1, s1, wc);
  }
  if (r < m) {
    const double* g0 = G + (size_t)r * gs;
    double s0 = 0;
    for (int c = lane; c < len; c += 32) s0 = fma(__ldg(g0 + c), wx[c], s0);
    s0 = warp_sum(s0);
    if (!ref) {
      const double ri = S.Ri[T.rioff[sd] + r];
      s0 = parked ? ri * (s0 - w[row0 + r]) : s0 - ri * w[row0 + r];
    } else if (vrow != nullptr && lane == 0) {
      vrow[row0 + r] = s0;
    }
    wc = fma(s0, s0, wc);
  }
  if (lane == 0) S.llcomp[sd] = (double)m * kHl2pi - 0.5 * wc;
}
cudaError_t launch_llw(const DevTree& T, const DevSlots& D, int rel, int slot0, int nslots, const double* w, int maxlen, cudaStream_t st,
                       double* vrow, int parked) {
  if (nslots <= 0) return cudaSuccess;
  const int wpb = kLlwThreads / 32;
  maxlen = (maxlen + 1) & ~1;
  const size_t smem = (size_t)wpb * maxlen * sizeof(double);
  static SmemOptIn optin;
  {
    cudaError_t e = ensure_dynamic_smem(llw_kernel, smem, optin);
    if (e != cudaSuccess) return e;
  }
  llw_kernel<<<(nslots + wpb - 1) / wpb, kLlwThreads, smem, st>>>(T, D, rel, slot0, nslots, w, maxlen, vrow, parked);
  return cudaGetLastError();
}

// Sum of the per-block log-density pieces (:987-988 / :815-816), in two parts so that a partitioned run can count the
// replicated blocks once and all-reduce the rest: part 0 = blocks [0, n_top) -> out[0..2], part 1 = [n_top, n) -> out[4..6];
// out[.] = {sum(logdet) + sum(llcomp), sum(logdet), 0 / *fail}.  kRedBlocks CTAs per part sum fixed chunks, the last CTA to
// finish adds the partial sums in chunk order: the summation order is fixed, the result deterministic run to run.
constexpr int kRedBlocks = 32;
__global__ void __launch_bounds__(256) loglik_reduce_kernel(DevSlots D, int rel, int n_top, int n, int* __restrict__ fail,
                                                            double* __restrict__ out, double* __restrict__ partial,
                                                            unsigned int* __restrict__ counter) {
  const int nblk = gridDim.x;  // CTAs per part: kRedBlocks, or 1 for a small tree (one CTA sums a part: no second stage to wait for)
  __shared__ double sa[256], sb[256];
  __shared__ bool last;
  const DevSlot S = pick_slot(D, D.chain->cur ^ rel);
  const int part = blockIdx.y, first = part ? n_top : 0, cnt = (part ? n : n_top) - first;
  const int chunk = (cnt + nblk - 1) / nblk;
  const int lo = first + blockIdx.x * chunk, hi = min(lo + chunk, first + cnt);
  double a = 0, b = 0;
  for (int i = lo + threadIdx.x; i < hi; i += 256) { a += S.logdet[i]; b += S.llcomp[i]; }
  sa[threadIdx.x] = a;
  sb[threadIdx.x] = b;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) { sa[threadIdx.x] += sa[threadIdx.x + s]; sb[threadIdx.x] += sb[threadIdx.x + s]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    partial[(part * kRedBlocks + blockIdx.x) * 2] = sa[0];
    partial[(part * kRedBlocks + blockIdx.x) * 2 + 1] = sb[0];
    if (nblk > 1) {
      __threadfence();
      last = atomicAdd(counter + part, 1u) == (unsigned)nblk - 1;
    } else {
      last = true;
    }
  }
  __syncthreads();
  if (last && threadIdx.x == 0) {
    __threadfence();
    double ta = 0, tb = 0;
    for (int k = 0; k < nblk; k++) { ta += partial[(part * kRedBlocks + k) * 2]; tb += partial[(part * kRedBlocks + k) * 2 + 1]; }
    double* o = out + 4 * part;
    o[0] = ta + tb;
    o[1] = ta;
    o[2] = 0.0;
    if (part && fail) { o[2] = (double)*fail; *fail = 0; }  // consumed and cleared: the counter is zero between BUILDs
    counter[part] = 0;  // ready for the next launch
  }
}
cudaError_t launch_loglik_reduce(const DevSlots& D, int rel, int n_top, int n, int* fail, double* out8, double* scratch,
                                 cudaStream_t st) {
  // scratch: 4 * kRedBlocks doubles of partial sums followed by two zero-initialised 32-bit counters
  // (the choice depends on the tree only: a handle always sums in the same order)
  loglik_reduce_kernel<<<dim3(n <= 8192 ? 1 : kRedBlocks, 2), 256, 0, st>>>(D, rel, n_top, n, fail, out8, scratch,
                                                            reinterpret_cast<unsigned int*>(scratch + 4 * kRedBlocks));
  return cudaGetLastError();
}

// partition only: sums of the messages of a replicated block's LOCAL children into its pseudo child, which is then
// all-reduced over the ranks (the replicated block pulls from the pseudo child like from any child)
__global__ void frontier_sum_kernel(DevTree T, const int* __restrict__ pseudo, const int* __restrict__ c0,
                                    const int* __restrict__ c1, const int* __restrict__ vlen, const int* __restrict__ ulen,
                                    double* __restrict__ V, double* __restrict__ U, int do_v, int do_u) {
  const int i = blockIdx.x, ps = pseudo[i];
  if (do_v)
    for (int e = threadIdx.x; e < vlen[i]; e += blockDim.x) {
      double s = 0;
      for (int c = c0[i]; c < c1[i]; c++) s += V[T.voff[c] + e];
      V[T.voff[ps] + e] = s;
    }
  if (do_u)
    for (int e = threadIdx.x; e < ulen[i]; e += blockDim.x) {
      double s = 0;
      for (int c = c0[i]; c < c1[i]; c++) s += U[T.uoff[c] + e];
      U[T.uoff[ps] + e] = s;
    }
}
cudaError_t launch_frontier_sum(const DevTree& T, int n, const int* pseudo, const int* c0, const int* c1, const int* vlen,
                                const int* ulen, double* V, double* U, int do_v, int do_u, cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  frontier_sum_kernel<<<n, 256, 0, st>>>(T, pseudo, c0, c1, vlen, ulen, V, U, do_v, do_u);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ prediction draws
// w_i = H_i w_pa + sqrt(K_ii - H_i Kxc_i) z_i  (:1306-1326); one thread per row of a prediction block
__global__ void predict_sample_kernel(DevTree T, int slot0, int nslots, const double* __restrict__ Hpred,
                                      const double* __restrict__ sdpred, double* __restrict__ w,
                                      const double* __restrict__ z) {
  const int sd = slot0 + blockIdx.x;
  const int m = T.m[sd], k = T.k[sd], coff = T.chain_off[sd], row0 = T.row0[sd];
  const double* H = Hpred + T.goff[sd];
  const int gs = T.gs[sd];
  const double* sdv = sdpred + T.rioff[sd];
  for (int r = threadIdx.x; r < m; r += blockDim.x) {
    double s = 0;
    for (int j = 0; j < k; j++) {
      const int a = T.chain[coff + j], mj = T.m[a], ar0 = T.row0[a];
      const double* h = H + (size_t)r * gs + T.chain_poff[coff + j];
      for (int pp = 0; pp < mj; pp++) s = fma(h[pp], w[ar0 + pp], s);
    }
    w[row0 + r] = s + sdv[r] * z[row0 + r];
  }
}
cudaError_t launch_predict_sample(const DevTree& T, int slot0, int nslots, const double* Hpred, const double* sdpred,
                                  double* w, const double* z, cudaStream_t st) {
  if (nslots <= 0) return cudaSuccess;
  predict_sample_kernel<<<nslots, 64, 0, st>>>(T, slot0, nslots, Hpred, sdpred, w, z);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ row kernels
// Philox4x32-10 -> two normals per call by Box-Muller
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
  const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
  const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
  c[0] = hi1 ^ c[1] ^ k0; c[1] = lo1; c[2] = hi0 ^ c[3] ^ k1; c[3] = lo0;
}
__device__ __forceinline__ void philox4x32(uint32_t (&c)[4], uint64_t seed) {
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; r++) { philox_round(c, k0, k1); k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
}
__device__ __forceinline__ double u01(uint32_t hi, uint32_t lo) { return ((((uint64_t)hi << 32 | lo) >> 11) + 0.5) * (1.0 / 9007199254740992.0); }
// one standard normal / one uniform for (seed, key, counter): Philox4x32-10 + Box-Muller
__device__ __forceinline__ double philox_normal(uint64_t seed, unsigned long long key, uint64_t counter) {
  uint32_t c[4] = {(uint32_t)key, (uint32_t)(key >> 32), (uint32_t)counter, (uint32_t)(counter >> 32)};
  philox4x32(c, seed);
  double sn, cs;
  sincospi(2.0 * u01(c[2], c[3]), &sn, &cs);
  return sqrt(-2.0 * log(u01(c[0], c[1]))) * cs;
}
__device__ __forceinline__ double philox_uniform(uint64_t seed, unsigned long long key, uint64_t counter) {
  uint32_t c[4] = {(uint32_t)key, (uint32_t)(key >> 32), (uint32_t)counter, (uint32_t)(counter >> 32)};
  philox4x32(c, seed);
  return u01(c[0], c[1]);
}
// streams of the chain's scalar draws: key = kStream* + index, counter = iteration (row streams use key = row id < 2^40)
constexpr unsigned long long kStreamU = 1ULL << 48, kStreamAccept = 2ULL << 48, kStreamGamma = 3ULL << 48, kStreamBeta = 4ULL << 48;
constexpr uint64_t kCounterYhat = 1ULL << 62;  // yhat noise: same row keys as the Gibbs normals, disjoint counters

__global__ void normals_kernel(double* __restrict__ z, long long n, uint64_t seed, uint64_t counter,
                               const long long* __restrict__ rowkey, const int* __restrict__ iter_ptr) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  // keyed by the row's id in the whole problem: the same draw whatever the partition (and on every rank that holds the row)
  z[i] = philox_normal(seed, (unsigned long long)rowkey[i], counter + (iter_ptr ? (uint64_t)*iter_ptr : 0));
}
cudaError_t launch_normals(double* z, long long n, uint64_t seed, uint64_t counter, const long long* rowkey, const int* iter_ptr,
                           cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  normals_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(z, n, seed, counter, rowkey, iter_ptr);
  return cudaGetLastError();
}

// sufficient statistics of the beta and tausq steps over the observed rows, per outcome j:
//   stat[j*(p+1) + a] = sum X(i,a) * (y_i - w[widx_i])   a < p     (X_available' (y_available - w), :1374-1375)
//   stat[j*(p+1) + p] = sum (y_i - XB_i - w_i)^2                   (bcore, :1399-1400)
// Stage 1 writes one partial vector per block, stage 2 adds the partials in block order (deterministic).
__global__ void __launch_bounds__(256) rowstats_kernel(DevTree T, const int* __restrict__ widx, long long n_all, int p,
                                                       int q, const double* __restrict__ w,
                                                       const double* __restrict__ xb, double* __restrict__ partial) {
  __shared__ double red[8];
  const int nv = q * (p + 1);
  double acc[kMaxStats];
  for (int v = 0; v < nv; v++) acc[v] = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_all; i += (long long)gridDim.x * blockDim.x) {
    const int wi = widx[i];
    if (wi < 0) continue;
    const int j = T.mvq[i];
    const double yi = T.y[i];
    const double res = yi - w[wi];
    for (int a = 0; a < p; a++) acc[j * (p + 1) + a] += T.X[i + (size_t)a * n_all] * res;
    const double e = yi - xb[i] - w[i];
    acc[j * (p + 1) + p] += e * e;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int v = 0; v < nv; v++) {
    const double s = warp_sum(acc[v]);
    if (lane == 0) red[warp] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0;
      for (int k2 = 0; k2 < 8; k2++) t += red[k2];
      partial[(size_t)blockIdx.x * nv + v] = t;
    }
    __syncthreads();
  }
}
// one CTA per statistic: the partial sums of the stage-1 blocks in a fixed order (deterministic)
__global__ void __launch_bounds__(128) rowstats_final_kernel(const double* __restrict__ partial, int nblocks, int nv, double* __restrict__ out) {
  __shared__ double red[128];
  const int v = blockIdx.x;
  double s = 0;
  for (int b = threadIdx.x; b < nblocks; b += 128) s += partial[(size_t)b * nv + v];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 64; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[v] = red[0];
}
cudaError_t launch_rowstats(const DevTree& T, const int* widx, long long n_all, int p, int q, const double* w,
                            const double* xb, double* partial, int nblocks, double* out, cudaStream_t st) {
  rowstats_kernel<<<nblocks, 256, 0, st>>>(T, widx, n_all, p, q, w, xb, partial);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  rowstats_final_kernel<<<q * (p + 1), 128, 0, st>>>(partial, nblocks, q * (p + 1), out);
  return cudaGetLastError();
}

// XB(i) = X(i,:) Bcoeff(:, mv_i)  (:1382)
__global__ void xb_kernel(DevTree T, long long n_all, int p, const double* __restrict__ bcoeff, double* __restrict__ xb) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_all) return;
  const int j = T.mvq[i];
  double s = 0;
  for (int a = 0; a < p; a++) s += T.X[i + (size_t)a * n_all] * bcoeff[a + j * p];
  xb[i] = s;
}
cudaError_t launch_xb(const DevTree& T, long long n_all, int p, const double* bcoeff, double* xb, cudaStream_t st) {
  xb_kernel<<<(unsigned)((n_all + 255) / 256), 256, 0, st>>>(T, n_all, p, bcoeff, xb);
  return cudaGetLastError();
}

// gather / scatter between boundary order and node-major order
__global__ void permute_kernel(const double* __restrict__ src, double* __restrict__ dst, const long long* __restrict__ map,
                               long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[map[i]];
}
cudaError_t launch_permute(const double* src, double* dst, const long long* map, long long n, cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  permute_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(src, dst, map, n);
  return cudaGetLastError();
}

// CrossCovarianceAG10 (covariance_functions.cpp:301-355): out(i,j), column-major n1 x n2
__global__ void crosscov_kernel(const double* __restrict__ x1, const double* __restrict__ y1, const int* __restrict__ q1,
                                long long n1, const double* __restrict__ x2, const double* __restrict__ y2,
                                const int* __restrict__ q2, long long n2, CovTab tab, double* __restrict__ out) {
  __shared__ CovTabS ct;
  load_covtab(ct, tab);
  __syncthreads();
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n1 * n2) return;
  const long long i = e % n1, j = e / n1;
  out[e] = cov_eval(ct, x1[i], y1[i], q1[i], x2[j], y2[j], q2[j]);
}
cudaError_t launch_crosscov(const double* x1, const double* y1, const int* q1, long long n1, const double* x2,
                            const double* y2, const int* q2, long long n2, const CovTab& tab, double* out,
                            cudaStream_t st) {
  const long long n = n1 * n2;
  if (n <= 0) return cudaSuccess;
  crosscov_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x1, y1, q1, n1, x2, y2, q2, n2, tab, out);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ device-resident chain
// The steps of spamtree_fit.cpp:203-289 and :376-389 that the reference runs on the host between the model-layer calls,
// as one-CTA kernels over the chain state in device memory (st_chain.hpp).  The arithmetic is st_mh.hpp's, the same
// functions the host path (and, through it, the pin against the reference's mh_adapt.h) uses.

// U ~ N(0, I), theta' = back(fwd(theta) + paramsd U) clipped (spamtree_fit.cpp:211-215) -> theta and covariance table of the
// alter slot
// iter_offset = 1: the proposal of the NEXT iteration, drawn right after this iteration's accept step (before the tick)
__global__ void mh_propose_kernel(ChainDev* C, int iter_offset) {
  const int npar = C->npar, cur = C->cur, alt = cur ^ 1;
  for (int j = threadIdx.x; j < npar; j += blockDim.x) C->U[j] = philox_normal(C->seed, kStreamU + j, (uint64_t)(C->iter + iter_offset));
  __syncthreads();
  if (threadIdx.x == 0) {
    mh_propose(npar, C->theta[cur], C->bounds, C->paramsd, C->U, C->theta[alt]);
    make_covtab_hd(C->theta[alt], npar, C->q, C->tab[alt]);
  }
}
cudaError_t launch_mh_propose(ChainDev* C, cudaStream_t st, int iter_offset) {
  mh_propose_kernel<<<1, 64, 0, st>>>(C, iter_offset);
  return cudaGetLastError();
}

// spamtree_fit.cpp:223-285: log-densities from the two reductions, Jacobian, accept decision, slot swap, RAM adaptation
// stage = 1: the adaptation's matrices (paramsd, prodparam, 2 npar^2 of scratch, U) are staged in shared memory — one thread
// runs a chain of dependent read-modify-writes over them, which in global memory is a chain of L2 round trips
__global__ void mh_accept_kernel(ChainDev* C, int mode, int have_llw, int stage) {
  extern __shared__ double acc_smem[];
  const int npar = C->npar, n2 = npar * npar;
  const bool adapt = mode == 0 && C->adapting;
  double *sp = C->paramsd, *pp = C->prodparam, *sc = C->scratch;
  const double* su = C->U;
  if (stage && adapt) {
    sp = acc_smem; pp = sp + n2; sc = pp + n2;
    double* u = sc + 2 * n2;
    for (int e = threadIdx.x; e < n2; e += blockDim.x) { sp[e] = C->paramsd[e]; pp[e] = C->prodparam[e]; }
    for (int e = threadIdx.x; e < npar; e += blockDim.x) u[e] = C->U[e];
    su = u;
    __syncthreads();
  }
  // the Jacobian's terms (four logarithms each) and the uniform draw by separate threads; thread 0 adds the terms in
  // mh_jacobian's order (st_mh.hpp), so the sum is the same
  __shared__ double s_term[kMaxPar];
  __shared__ double s_u;
  if (mode == 0) {
    const int cur0 = C->cur, alt0 = cur0 ^ 1;
    for (int j = threadIdx.x; j < npar; j += blockDim.x) {
      const double lo = C->bounds[j], hi = C->bounds[j + npar], pj = C->theta[cur0][j], nj = C->theta[alt0][j];
      s_term[j] = (-log(hi - pj) - log(pj - lo)) - (-log(hi - nj) - log(nj - lo));
    }
    if (threadIdx.x == blockDim.x - 1) s_u = philox_uniform(C->seed, kStreamAccept, (uint64_t)C->iter);
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const int cur = C->cur, alt = cur ^ 1, m = C->iter;
    if (have_llw) { C->loglik[cur] = C->red_llw[0] + C->red_llw[4]; C->logdet[cur] = C->red_llw[1] + C->red_llw[5]; }
    const bool acceptable = C->red_build[6] == 0.0;
    if (acceptable) {  // on failure the reference leaves the alter slot's log-density untouched (:971-982)
      C->loglik[alt] = C->red_build[0] + C->red_build[4];
      C->logdet[alt] = C->red_build[1] + C->red_build[5];
    } else {
      C->n_chol_fail++;
    }
    const double new_loglik = C->loglik[alt], current_loglik = C->loglik[cur];
    if (isnan(current_loglik)) C->nan_loglik = 1;  // spamtree_fit.cpp:234-237
    bool accepted;
    double logaccept = 0.0;
    if (mode == 0) {
      double jac = 0;
      for (int j = 0; j < npar; j++) jac += s_term[j];
      logaccept = new_loglik - current_loglik + jac;
      const double u = s_u;
      C->last_logaccept = logaccept; C->last_u = u;
      accepted = (u < mh_accept_prob(logaccept)) && acceptable;
    } else {
      accepted = (mode == 1) && acceptable;
    }
    if (accepted) {
      C->n_accepted++;
      C->cur = alt;  // accept_make_change (:1432-1435): the kernels that follow read the new slot
      C->pred_valid = 0;
    }
    C->accepted_now = accepted ? 1 : 0;
    if (adapt)  // :285 (a failed chol(S) keeps the previous factor and is counted)
      if (!ram_adapt(npar, sp, pp, &C->ram_started, su, (acceptable ? 1.0 : 0.0) * exp(logaccept), m, sc))
        C->n_ram_fail++;
  }
  if (stage && adapt) {
    __syncthreads();
    for (int e = threadIdx.x; e < n2; e += blockDim.x) { C->paramsd[e] = sp[e]; C->prodparam[e] = pp[e]; }
  }
}
cudaError_t launch_mh_accept(ChainDev* C, int mode, int have_llw, cudaStream_t st, int npar) {
  const size_t smem = ((size_t)4 * npar * npar + npar) * sizeof(double);
  const int stage = npar > 0 && smem <= 40 * 1024;
  mh_accept_kernel<<<1, 64, stage ? smem : 0, st>>>(C, mode, have_llw, stage);
  return cudaGetLastError();
}

// need_update = any |param - predict_param| > 1e-05 (spamtree_fit.cpp:300); predict_param <- param (:305)
__global__ void predict_gate_kernel(ChainDev* C) {
  if (threadIdx.x != 0) return;
  const double* th = C->theta[C->cur];
  bool need = !C->pred_valid;
  for (int j = 0; j < C->npar; j++) {
    if (fabs(th[j] - C->predict_param[j]) > 1e-05) need = true;
    C->predict_param[j] = th[j];
  }
  C->predict_build = need ? 1 : 0;
  C->pred_valid = 1;
}
cudaError_t launch_predict_gate(ChainDev* C, cudaStream_t st) {
  predict_gate_kernel<<<1, 32, 0, st>>>(C);
  return cudaGetLastError();
}

// Marsaglia-Tsang gamma(shape >= 1, scale) on a Philox stream (the host path's HostRng::gamma, st_common.hpp)
// x0, u0: the first attempt's normal and uniform, drawn by other threads (same streams: same value)
__device__ inline double philox_gamma(uint64_t seed, unsigned long long key, uint64_t counter, double shape, double scale, double x0, double u0) {
  const double d = shape - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
  for (unsigned long long att = 0;; att++) {
    const double x = att ? philox_normal(seed, key + (att << 8), counter) : x0;
    double v = 1.0 + c * x;
    if (v <= 0) continue;
    v = v * v * v;
    const double u = att ? philox_uniform(seed, key + (att << 8) + 128, counter) : u0;
    if (u < 1.0 - 0.0331 * x * x * x * x) return d * v * scale;
    if (log(u) < 0.5 * x * x + d * (1.0 - v + log(v))) return d * v * scale;
  }
}
// gibbs_sample_tausq (spamtree_model.cpp:1393-1417) then gibbs_sample_beta (:1364-1391), one thread per outcome.
// stats[j*(p+1) + a] = X_j'(y - w)_a, stats[j*(p+1) + p] = |y - XB - w|^2 over the outcome's observed rows (rowstats_kernel)
__global__ void tausq_beta_kernel(ChainDev* C, const double* __restrict__ stats, const double* __restrict__ xtx,
                                  double* __restrict__ tausq_inv, double* __restrict__ bcoeff, double* __restrict__ scratch,
                                  int sample_tausq, int sample_beta, int stage) {
  extern __shared__ double tb_smem[];  // stage = 1: the p x p work arrays of every outcome (else `scratch` in global memory)
  if (stage) scratch = tb_smem;
  const int j = threadIdx.x, p = C->p, q = C->q;
  const uint64_t it = (uint64_t)C->iter;
  // every draw by a thread of its own (a normal is a Philox block, a logarithm, a square root and a sincospi: the one thread
  // per outcome that used to draw p + 2 of them in sequence spent most of its time there)
  __shared__ double s_zb[kMaxStats], s_gx[kMaxQ], s_gu[kMaxQ];
  const bool par_draws = q * p <= kMaxStats;
  if (par_draws) {
    const int nz = sample_beta ? q * p : 0, ng = sample_tausq ? q : 0;
    for (int t = threadIdx.x; t < nz + 2 * ng; t += blockDim.x) {
      if (t < nz) s_zb[t] = philox_normal(C->seed, kStreamBeta + ((unsigned long long)(t / p) << 32) + (t % p), it);
      else if (t < nz + ng) s_gx[t - nz] = philox_normal(C->seed, kStreamGamma + ((unsigned long long)(t - nz) << 32), it);
      else s_gu[t - nz - ng] = philox_uniform(C->seed, kStreamGamma + ((unsigned long long)(t - nz - ng) << 32) + 128, it);
    }
    __syncthreads();
  }
  if (j >= q) return;
  if (sample_tausq) {
    const double bcore = stats[j * (p + 1) + p];
    const unsigned long long gk = kStreamGamma + ((unsigned long long)j << 32);
    const double x0 = par_draws ? s_gx[j] : philox_normal(C->seed, gk, it), u0 = par_draws ? s_gu[j] : philox_uniform(C->seed, gk + 128, it);
    tausq_inv[j] = philox_gamma(C->seed, gk, it, 2.01 + C->nobs[j] / 2.0, 1.0 / (1.0 + .5 * bcore), x0, u0);
  }
  if (sample_beta) {
    const double tq = tausq_inv[j];
    double* Si = scratch + (size_t)j * (2 * p * p + 4 * p);  // precision -> its Cholesky factor (column-major)
    double* Sc = Si + p * p;                                 // inverse of the factor
    double* v = Sc + p * p;                                  // xp | t | bmu | sz: 4 p doubles of the outcome's own
    for (int a = 0; a < p; a++)
      for (int b = 0; b < p; b++) Si[a + b * p] = tq * xtx[(size_t)j * p * p + (b <= a ? b + a * p : a + b * p)] + (a == b ? .01 : 0.0);  // symmatu; Vi = .01 I (:157)
    if (!mh_chol_lower(Si, p)) { C->gibbs_fail = 1; return; }
    for (int c = 0; c < p; c++) {  // Sc = Si^-1 (lower)
      for (int r = 0; r < c; r++) Sc[r + c * p] = 0.0;
      Sc[c + c * p] = 1.0 / Si[c + c * p];
      for (int r = c + 1; r < p; r++) {
        double s = 0;
        for (int k = c; k < r; k++) s += Si[r + k * p] * Sc[k + c * p];
        Sc[r + c * p] = -s / Si[r + r * p];
      }
    }
    double *xp = v, *t = v + p, *bmu = v + 2 * p;
    for (int a = 0; a < p; a++) xp[a] = tq * stats[j * (p + 1) + a];  // Vim = 0 (:158-159)
    for (int a = 0; a < p; a++) { double s = 0; for (int b = 0; b <= a; b++) s += Sc[a + b * p] * xp[b]; t[a] = s; }
    for (int a = 0; a < p; a++) { double s = 0; for (int b = a; b < p; b++) s += Sc[b + a * p] * t[b]; bmu[a] = s; }
    for (int a = 0; a < p; a++) xp[a] = par_draws ? s_zb[j * p + a] : philox_normal(C->seed, kStreamBeta + ((unsigned long long)j << 32) + a, it);
    for (int a = 0; a < p; a++) {
      double s = 0;
      for (int b = a; b < p; b++) s += Sc[b + a * p] * xp[b];
      bcoeff[a + j * p] = bmu[a] + s;
    }
  }
}
cudaError_t launch_tausq_beta(ChainDev* C, const double* stats, const double* xtx, double* tausq_inv, double* bcoeff,
                              double* scratch, int sample_tausq, int sample_beta, cudaStream_t st, int p, int q) {
  const size_t smem = (size_t)q * (2 * p * p + 4 * p) * sizeof(double);  // the layout of `scratch`
  const int stage = p > 0 && smem <= 40 * 1024;
  tausq_beta_kernel<<<1, 64, stage ? smem : 0, st>>>(C, stats, xtx, tausq_inv, bcoeff, scratch, sample_tausq, sample_beta, stage);
  return cudaGetLastError();
}

// save (spamtree_fit.cpp:376-382): column msaved of theta_mcmc (npar x keep), tausq_mcmc (q x keep), beta_mcmc (p x keep x q)
__global__ void record_kernel(ChainDev* C, const double* __restrict__ tausq_inv, const double* __restrict__ bcoeff,
                              double* __restrict__ theta_mcmc, double* __restrict__ beta_mcmc, double* __restrict__ tausq_mcmc, int keep,
                              int tick) {
  const int ms = C->msaved, npar = C->npar, p = C->p, q = C->q;
  if (ms < keep) {
    for (int j = threadIdx.x; j < npar; j += blockDim.x) theta_mcmc[j + (size_t)ms * npar] = C->theta[C->cur][j];
    for (int j = threadIdx.x; j < q; j += blockDim.x) tausq_mcmc[j + (size_t)ms * q] = 1.0 / tausq_inv[j];
    for (int e = threadIdx.x; e < p * q; e += blockDim.x) { const int a = e % p, j = e / p; beta_mcmc[a + (size_t)ms * p + (size_t)j * p * keep] = bcoeff[e]; }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    C->msaved = ms + 1;
    if (tick) C->iter++;  // (the end of a saved iteration: chain_tick_kernel's work rides along)
  }
}
cudaError_t launch_record(ChainDev* C, const double* tausq_inv, const double* bcoeff, double* theta_mcmc, double* beta_mcmc,
                          double* tausq_mcmc, int keep, cudaStream_t st, int tick) {
  record_kernel<<<1, 64, 0, st>>>(C, tausq_inv, bcoeff, theta_mcmc, beta_mcmc, tausq_mcmc, keep, tick);
  return cudaGetLastError();
}

// yhat = XB + w + tausq_inv^(-1/2) N(0,1), boundary order (spamtree_fit.cpp:384); iperm: boundary row -> node-major row
__global__ void yhat_kernel(DevTree T, const double* __restrict__ w, const double* __restrict__ xb, const double* __restrict__ tausq_inv,
                            const long long* __restrict__ iperm, const long long* __restrict__ rowkey, long long n, const ChainDev* C,
                            double* __restrict__ out) {
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n) return;
  const long long i = iperm[b];
  const double e = philox_normal(C->seed, (unsigned long long)rowkey[i], kCounterYhat + (uint64_t)C->iter);
  out[b] = xb[i] + w[i] + rsqrt(tausq_inv[T.mvq[i]]) * e;
}
cudaError_t launch_yhat(const DevTree& T, const double* w, const double* xb, const double* tausq_inv, const long long* iperm,
                        const long long* rowkey, long long n, const ChainDev* C, double* out, cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  yhat_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(T, w, xb, tausq_inv, iperm, rowkey, n, C, out);
  return cudaGetLastError();
}

__global__ void chain_set_theta_kernel(ChainDev* C, int rel, const __grid_constant__ ThetaPack P) {
  const int phys = C->cur ^ rel;
  for (int j = threadIdx.x; j < P.n; j += blockDim.x) C->theta[phys][j] = P.theta[j];
  // (the table word by word, by all threads: CovTab is an int followed by doubles, 8-byte aligned)
  const unsigned long long* src = reinterpret_cast<const unsigned long long*>(&P.tab);
  unsigned long long* dst = reinterpret_cast<unsigned long long*>(&C->tab[phys]);
  for (int j = threadIdx.x; j < (int)(sizeof(CovTab) / 8); j += blockDim.x) dst[j] = src[j];
}
cudaError_t launch_chain_set_theta(ChainDev* C, int rel, const ThetaPack& pack, cudaStream_t st) {
  chain_set_theta_kernel<<<1, 64, 0, st>>>(C, rel, pack);
  return cudaGetLastError();
}
__global__ void chain_flip_kernel(ChainDev* C) { C->cur ^= 1; C->pred_valid = 0; }
cudaError_t launch_chain_flip(ChainDev* C, cudaStream_t st) {
  chain_flip_kernel<<<1, 1, 0, st>>>(C);
  return cudaGetLastError();
}
__global__ void chain_tick_kernel(ChainDev* C) { C->iter++; }
cudaError_t launch_chain_tick(ChainDev* C, cudaStream_t st) {
  chain_tick_kernel<<<1, 1, 0, st>>>(C);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ predict_new
// normals of the draws at new rows: key = stream + row (the caller's index of the new row), counter = position of the sample
// in the call — the same numbers whatever the launch shape or the layout of the rows into pseudo-blocks
constexpr unsigned long long kStreamPredW = 5ULL << 48, kStreamPredY = 6ULL << 48;

// w of sample b of a staged block (element (row, b) at src[row * si + b * sb], boundary order) -> node-major order
__global__ void gather_sample_kernel(const double* __restrict__ src, long long si, long long sb, int b, const long long* __restrict__ perm,
                                     double* __restrict__ dst, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[perm[i] * si + (long long)b * sb];
}
cudaError_t launch_gather_sample(const double* src, long long si, long long sb, int b, const long long* perm, double* dst, long long n,
                                 cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  gather_sample_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(src, si, sb, b, perm, dst, n);
  return cudaGetLastError();
}

// w_new = mean + sd z, y_new = x' beta[:, mv] + w_new + sqrt(tausq[mv]) eps (spamtree_fit.cpp:384), one thread per new row;
// the running mean / sum of squared deviations of both over the samples of the call (Welford, FP64, in sample order)
__global__ void predict_draw_kernel(long long n, const long long* __restrict__ lay2row, const int* __restrict__ mvq,
                                    const double* __restrict__ X, int p, const double* __restrict__ mean, const double* __restrict__ sd,
                                    const __grid_constant__ PredDrawPack pk, uint64_t seed, int j, const double* __restrict__ z,
                                    const double* __restrict__ eps, double* __restrict__ wout, double* __restrict__ yout,
                                    double* __restrict__ mout, double* __restrict__ sdout, double* __restrict__ acc) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const long long i = lay2row[k];
  const int qi = mvq[i];
  const double zz = z ? z[i] : philox_normal(seed, kStreamPredW + (unsigned long long)i, (uint64_t)j);
  const double ee = eps ? eps[i] : philox_normal(seed, kStreamPredY + (unsigned long long)i, (uint64_t)j);
  const double wv = mean[k] + sd[k] * zz;
  double xb = 0;
  if (X)
    for (int a = 0; a < p; a++) xb += X[i + (size_t)a * n] * pk.beta[a + qi * p];
  const double yv = xb + wv + pk.sdtau[qi] * ee;
  wout[i] = wv;
  yout[i] = yv;
  if (mout) mout[i] = mean[k];
  if (sdout) sdout[i] = sd[k];
  const double cnt = (double)(j + 1);
  double* a = acc + 4 * i;  // {mean w, M2 w, mean y, M2 y}
  if (j == 0) { a[0] = wv; a[1] = 0.0; a[2] = yv; a[3] = 0.0; return; }
  const double dw = wv - a[0];
  a[0] += dw / cnt;
  a[1] += dw * (wv - a[0]);
  const double dy = yv - a[2];
  a[2] += dy / cnt;
  a[3] += dy * (yv - a[2]);
}
cudaError_t launch_predict_draw(long long n, const long long* lay2row, const int* mvq, const double* X, int p, const double* mean,
                                const double* sd, const PredDrawPack& pk, uint64_t seed, int j, const double* z, const double* eps,
                                double* wout, double* yout, double* mout, double* sdout, double* acc, cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  predict_draw_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, lay2row, mvq, X, p, mean, sd, pk, seed, j, z, eps, wout, yout, mout,
                                                                   sdout, acc);
  return cudaGetLastError();
}
// per-row summaries of the call's S samples: mean and sd (ddof = 1; 0 for one sample) of w_new and y_new
__global__ void predict_moments_kernel(long long n, int S, const double* __restrict__ acc, double* __restrict__ out4) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double* a = acc + 4 * i;
  out4[i] = a[0];
  out4[n + i] = S > 1 ? sqrt(a[1] / (S - 1)) : 0.0;
  out4[2 * n + i] = a[2];
  out4[3 * n + i] = S > 1 ? sqrt(a[3] / (S - 1)) : 0.0;
}
cudaError_t launch_predict_moments(long long n, int S, const double* acc, double* out4, cudaStream_t st) {
  if (n <= 0 || S <= 0) return cudaSuccess;
  predict_moments_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, S, acc, out4);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ summaries of stored draws
// Doubles as 64-bit keys whose unsigned order is the numeric order (negative: all bits flipped; otherwise: sign bit set)
__device__ __forceinline__ unsigned long long summary_key(double x) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(x);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ULL);
}
__device__ __forceinline__ double summary_val(unsigned long long k) {
  return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffULL) : ~k));
}

// sum over the G threads of each row group (threads [r G, (r + 1) G)), pairwise in a fixed order; every thread gets its
// group's total.  red: blockDim.x doubles.  Called by every thread of the CTA.
__device__ __forceinline__ double summary_group_sum(double v, double* red, int G) {
  const int t = threadIdx.x, lane = t % G;
  red[t] = v;
  __syncthreads();
  for (int s = G >> 1; s > 0; s >>= 1) {
    if (lane < s) red[t] += red[t + s];
    __syncthreads();
  }
  const double total = red[t - lane];
  __syncthreads();
  return total;
}

// sort each of the R rows of S keys at key[r S ..) ascending: the all-ascending form of the bitonic network (a "flip" stage
// then half-cleaners) over pairs (i, j > i), so positions >= S act as +inf and are never touched (no padding is staged).
// Called by every thread of the CTA; ends with a barrier.
__device__ void summary_sort_rows(unsigned long long* key, int R, int S) {
  const int t = threadIdx.x, T = blockDim.x;
  int P2 = 1;
  while (P2 < S) P2 <<= 1;
  const int half = P2 >> 1;
  const long long pairs = (long long)R * half;
  for (int k = 2; k <= P2; k <<= 1) {
    for (int d = k >> 1; d > 0; d >>= 1) {
      const bool flip = d == (k >> 1);
      for (long long e = t; e < pairs; e += T) {
        const int rr = (int)(e / half), pp = (int)(e % half);
        const int i = (pp / d) * 2 * d + pp % d;
        const int j = flip ? (i ^ (k - 1)) : i + d;
        if (j < S) {
          unsigned long long* kk = key + (long long)rr * S;
          const unsigned long long a = kk[i], c = kk[j];
          if (a > c) { kk[i] = c; kk[j] = a; }
        }
      }
      __syncthreads();
    }
  }
}

// the p-quantile of S sorted keys: numpy's method "linear" (R type 7) with its virtual-index and _lerp formulas, without
// contraction
__device__ double summary_quantile(const unsigned long long* kk, int S, double p) {
  const double vi = __dmul_rn((double)(S - 1), p);
  if (vi >= (double)(S - 1)) return summary_val(kk[S - 1]);
  const int lo = (int)floor(vi);
  const double g = __dsub_rn(vi, (double)lo);
  const double a = summary_val(kk[lo]), c = summary_val(kk[lo + 1]);
  const double diff = __dsub_rn(c, a);
  return g >= 0.5 ? __dsub_rn(c, __dmul_rn(diff, __dsub_rn(1.0, g))) : __dadd_rn(a, __dmul_rn(diff, g));
}

// One CTA per tile of R rows of a [sample][row] store (element (s, i) at src[s * n + i]).  The tile's S x R values are read
// once with coalesced loads (consecutive threads, consecutive rows), staged as order-preserving keys (row-major: key[r S + s]),
// and every statistic is formed from the staged copy: the moments and batch means in sample order, then the quantiles after a
// bitonic sort of each row in shared memory (summary_sort_rows).  Every reduction is over G = T / R
// threads per row in a fixed order.  Outputs: mean, sd (ddof 1), quant (n x np, column-major), mcse, ess (batch means).
__global__ void __launch_bounds__(kSummaryThreads)
summary_kernel(const double* __restrict__ src, long long n, int S, int R, const double* __restrict__ probs, int np,
               double* __restrict__ mean_out, double* __restrict__ sd_out, double* __restrict__ quant, double* __restrict__ mcse_out,
               double* __restrict__ ess_out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* red = reinterpret_cast<double*>(smem_raw);                                 // T doubles
  unsigned long long* key = reinterpret_cast<unsigned long long*>(red + blockDim.x);  // R x S keys
  const int T = blockDim.x, t = threadIdx.x, G = T / R, r = t / G, lane = t % G;
  const long long row0 = (long long)blockIdx.x * R;
  const int nr = (int)min((long long)R, n - row0);
  // ---- stage: element e of the tile is (sample e / R, row e % R)
  const long long tot = (long long)S * R;
  for (long long e = t; e < tot; e += T) {
    const int s = (int)(e / R), rr = (int)(e % R);
    key[(long long)rr * S + s] = rr < nr ? summary_key(src[(long long)s * n + row0 + rr]) : 0ULL;
  }
  __syncthreads();
  const unsigned long long* kr = key + (long long)r * S;
  // ---- mean and sd (two passes over the staged row, in sample order per thread)
  double acc = 0.0;
  for (int s = lane; s < S; s += G) acc += summary_val(kr[s]);
  const double mean = summary_group_sum(acc, red, G) / S;
  acc = 0.0;
  for (int s = lane; s < S; s += G) { const double dv = summary_val(kr[s]) - mean; acc += dv * dv; }
  const double ss = summary_group_sum(acc, red, G);
  const double var = S > 1 ? ss / (S - 1) : 0.0;
  // ---- batch means: b = floor(sqrt(S)) draws per batch, B = floor(S / b) batches over the first B b draws
  int b = (int)sqrt((double)S);
  while ((long long)(b + 1) * (b + 1) <= S) b++;
  while (b > 1 && (long long)b * b > S) b--;
  const int B = S / b;
  acc = 0.0;
  for (int k = lane; k < B; k += G) {
    double bs = 0.0;
    for (int s = k * b; s < k * b + b; s++) bs += summary_val(kr[s]);
    acc += bs / b;
  }
  const double bmean = summary_group_sum(acc, red, G) / B;
  acc = 0.0;
  for (int k = lane; k < B; k += G) {
    double bs = 0.0;
    for (int s = k * b; s < k * b + b; s++) bs += summary_val(kr[s]);
    const double dv = bs / b - bmean;
    acc += dv * dv;
  }
  const double bss = summary_group_sum(acc, red, G);
  if (lane == 0 && r < nr) {
    const long long i = row0 + r;
    const double sig2 = B > 1 ? (double)b * (bss / (B - 1)) : 0.0;
    const bool ok = S >= 2 && sig2 > 0.0;
    mean_out[i] = mean;
    sd_out[i] = sqrt(var);
    mcse_out[i] = ok ? sqrt(sig2 / S) : __longlong_as_double(0x7ff8000000000000LL);
    ess_out[i] = ok ? (double)S * var / sig2 : __longlong_as_double(0x7ff8000000000000LL);
  }
  if (np == 0) return;
  summary_sort_rows(key, R, S);
  for (int e = t; e < R * np; e += T) {
    const int rr = e / np, jp = e % np;
    if (rr < nr) quant[row0 + rr + (long long)jp * n] = summary_quantile(key + (long long)rr * S, S, probs[jp]);
  }
}
int summary_rows_per_cta(int S, size_t smem_cap) {
  if (S < 1) return 0;
  const size_t avail = smem_cap - (size_t)kSummaryThreads * sizeof(double);
  int R = kSummaryMaxRows;
  while (R >= 1 && (size_t)R * S * sizeof(unsigned long long) > avail) R >>= 1;
  return R;
}
size_t summary_smem_bytes(int S, int R) { return (size_t)kSummaryThreads * sizeof(double) + (size_t)R * S * sizeof(unsigned long long); }
cudaError_t launch_summary(const double* src, long long n, int S, int R, const double* probs, int np, double* mean, double* sd, double* quant,
                           double* mcse, double* ess, cudaStream_t st) {
  if (n <= 0 || S <= 0) return cudaSuccess;
  static SmemOptIn opt;
  const size_t smem = summary_smem_bytes(S, R);
  cudaError_t e = ensure_dynamic_smem(summary_kernel, smem, opt);
  if (e != cudaSuccess) return e;
  summary_kernel<<<(unsigned)((n + R - 1) / R), kSummaryThreads, smem, st>>>(src, n, S, R, probs, np, mean, sd, quant, mcse, ess);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------ several chains: pooled summaries and
// rank-normalised split-R-hat, bulk-ESS and tail-ESS (st_summarize_chains / st_summarize_draws; DESIGN.md §5d)
typedef unsigned long long u64;
__device__ __forceinline__ int keys_lower(const u64* b, int N, u64 k) {  // first j with b[j] >= k
  int lo = 0, hi = N;
  while (lo < hi) { const int m = (lo + hi) >> 1; if (b[m] < k) lo = m + 1; else hi = m; }
  return lo;
}
__device__ __forceinline__ int keys_upper(const u64* b, int N, u64 k) {  // first j with b[j] > k
  int lo = 0, hi = N;
  while (lo < hi) { const int m = (lo + hi) >> 1; if (b[m] <= k) lo = m + 1; else hi = m; }
  return lo;
}

// One row of a tile: a = its K x S draws as keys in sample order (a[c S + s]), b = the same sorted, cm = 2K doubles of
// scratch.  Split chain c (of M = 2K, h draws each) is the first (c even) or the last (c odd) h draws of chain c / 2; for odd
// S each chain's middle draw a[c S + h] belongs to no split chain.
struct ChainsRow {
  u64* a;
  const u64* b;
  double* cm;
  int K, S, h, N;
  __device__ int pos(int c, int i) const { return (c >> 1) * S + ((c & 1) ? S - h : 0) + i; }
  __device__ bool odd() const { return S & 1; }
  __device__ u64 mid(int k) const { return a[k * S + h]; }
  // (count < v, count <= v) of the split draws: of all N from b, less the middle draws for odd S
  __device__ void rank_counts(u64 v, int& lt, int& le) const {
    lt = keys_lower(b, N, v);
    le = keys_upper(b, N, v);
    if (odd())
      for (int k = 0; k < K; k++) { const u64 m = mid(k); lt -= m < v; le -= m <= v; }
  }
  // the j-th smallest split draw (0-based): the first b[i] with more than j split draws <= b[i]
  __device__ double split_order_stat(int j) const {
    int lo = 0, hi = N - 1;
    while (lo < hi) {
      const int m = (lo + hi) >> 1;
      int lt, le;
      rank_counts(b[m], lt, le);
      if (le > j) hi = m; else lo = m + 1;
    }
    return summary_val(b[lo]);
  }
  // z-scale of a key among the 2 K h split draws: Phi^-1((r - 3/8) / (N' + 1/4)), r its average rank
  __device__ double z_bulk(u64 v) const {
    int lt, le;
    rank_counts(v, lt, le);
    return normcdfinv(((double)(lt + 1 + le) / 2.0 - 0.375) / ((double)(2 * K * h) + 0.25));
  }
  // z-scale of f = |x - med| among the folded split draws.  b[0, m) (values < med) folds to a non-increasing run and b[m, N)
  // to a non-decreasing one, so each count is a binary search on either side of m with the folded values formed on the fly
  // exactly as |x - med| is formed for x itself
  __device__ double z_fold(double f, double med, int m) const {
    int l0 = 0, l1 = m, r0 = m, r1 = N;  // l: first j < m with |b_j - med| < f; r: first j >= m with |b_j - med| >= f
    while (l0 < l1) { const int q = (l0 + l1) >> 1; if (fabs(summary_val(b[q]) - med) < f) l1 = q; else l0 = q + 1; }
    while (r0 < r1) { const int q = (r0 + r1) >> 1; if (fabs(summary_val(b[q]) - med) >= f) r1 = q; else r0 = q + 1; }
    int lt = r0 - l0;
    int u0 = 0, u1 = m, v0 = m, v1 = N;  // the same with <= f / > f
    while (u0 < u1) { const int q = (u0 + u1) >> 1; if (fabs(summary_val(b[q]) - med) <= f) u1 = q; else u0 = q + 1; }
    while (v0 < v1) { const int q = (v0 + v1) >> 1; if (fabs(summary_val(b[q]) - med) > f) v1 = q; else v0 = q + 1; }
    int le = v0 - u0;
    if (odd())
      for (int k = 0; k < K; k++) { const double g = fabs(summary_val(mid(k)) - med); lt -= g < f; le -= g <= f; }
    return normcdfinv(((double)(lt + 1 + le) / 2.0 - 0.375) / ((double)(2 * K * h) + 0.25));
  }
};

// Chain means of f(c, i) (c < M split chains, i < h) into row.cm, then every thread of the row gets mean_var (= W, the mean
// within-chain variance, ddof 1) and var_m (the variance of the chain means, ddof 1).  Every sum runs in a fixed order.
// Called by every thread of the CTA.
template <class F>
__device__ void chains_moments(const ChainsRow& row, F f, int G, int lane, double* red, double& mean_var, double& var_m) {
  const int M = 2 * row.K, h = row.h, t = threadIdx.x;
  const int tpc = max(1, G / M), cpp = G / tpc;  // threads per chain, chains per pass
  for (int c0 = 0; c0 < M; c0 += cpp) {
    const int c = c0 + lane / tpc, part = lane % tpc;
    const bool mine = lane / tpc < cpp && c < M;
    double acc = 0.0;
    if (mine)
      for (int i = part; i < h; i += tpc) acc += f(c, i);
    red[t] = acc;
    __syncthreads();
    if (mine && part == 0) {
      double s = 0.0;
      for (int j = 0; j < tpc; j++) s += red[t + j];
      row.cm[c] = s / h;
    }
    __syncthreads();
  }
  double acc = 0.0;
  for (long long e = lane; e < (long long)M * h; e += G) {
    const int c = (int)(e / h), i = (int)(e % h);
    const double d = f(c, i) - row.cm[c];
    acc += d * d;
  }
  const double ss = summary_group_sum(acc, red, G);
  mean_var = ss / ((double)M * h) * h / (h - 1);
  double mm = 0.0;
  for (int c = 0; c < M; c++) mm += row.cm[c];
  mm /= M;
  double vm = 0.0;
  for (int c = 0; c < M; c++) { const double d = row.cm[c] - mm; vm += d * d; }
  var_m = vm / (M - 1);
}

__device__ __forceinline__ double chains_rhat(double mean_var, double var_m, int h) {
  return mean_var > 0.0 ? sqrt(((double)h * var_m / mean_var + h - 1) / h) : __longlong_as_double(0x7ff8000000000000LL);
}

// ESS of f after chains_moments (row.cm holds its chain means): autocovariances by direct sums over lags, two lags per step,
// until Geyer's initial positive sequence stops (row by row; the CTA steps while any row goes on).  The initial monotone
// sequence is applied on the fly: it replaces each pair sum by the running minimum of the pair sums before it.
template <class F>
__device__ double chains_ess(const ChainsRow& row, F f, int G, int lane, double* red, double mean_var, double var_m, bool live) {
  const int M = 2 * row.K, h = row.h;
  const double var_plus = mean_var * (h - 1) / h + var_m;
  bool act = live && var_plus > 0.0;
  auto lag_mean = [&](int lag, bool on) {  // mean over the chains of the biased autocovariance at lag
    double acc = 0.0;
    if (on) {
      const int L = h - lag;
      for (long long e = lane; e < (long long)M * L; e += G) {
        const int c = (int)(e / L), i = (int)(e % L);
        acc += (f(c, i) - row.cm[c]) * (f(c, i + lag) - row.cm[c]);
      }
    }
    return summary_group_sum(acc, red, G) / h / M;
  };
  const double a1 = lag_mean(1, act);
  double ev = 1.0, od = act ? 1.0 - (mean_var - a1) / var_plus : 0.0;
  double pmin = 0.0, sum_p = 0.0, last = 0.0;
  for (int k = 0;; k++) {
    if (act) {  // pair k = (rho_2k, rho_2k+1): inside the sequence, or the pair that ends it
      const double P = ev + od;
      if (2 * k + 1 < h - 3 && P > 0.0) {
        pmin = k ? fmin(pmin, P) : P;
        sum_p += pmin;
      } else {
        last = (ev > 0.0 || P >= 0.0) ? ev : 0.0;
        act = false;
      }
    }
    if (!__syncthreads_or(act)) break;
    const double ae = lag_mean(2 * k + 2, act), ao = lag_mean(2 * k + 3, act);
    if (act) { ev = 1.0 - (mean_var - ae) / var_plus; od = 1.0 - (mean_var - ao) / var_plus; }
  }
  if (!(live && var_plus > 0.0)) return __longlong_as_double(0x7ff8000000000000LL);
  const double n = (double)M * h;
  const double tau = fmax(-1.0 + 2.0 * sum_p + last, 1.0 / log10(n));
  return n / tau;
}

// One CTA per tile of R rows; chain c's draws of row i at src[c][s n + i].  The tile's K S draws per row are read with
// coalesced loads into keys in sample order (a) and copied (b), -0 staged as +0; b is sorted (summary_sort_rows).  Pooled mean and sd come
// from a, pooled quantiles, q05 / q95 and the split median from b.  Then, in this order: tail-ESS of the indicators
// x <= q05 / q95 (read from a); the folded R-hat from z-scales formed on the fly; the bulk z-scales, written over a in place
// (each thread reads and writes only its own draws, and the middle draws for odd S stay keys); bulk R-hat and ESS.
__global__ void __launch_bounds__(kSummaryThreads)
chains_summary_kernel(const double* const* __restrict__ src, long long n, int K, int S, int R, const double* __restrict__ probs,
                      int np, double* __restrict__ mean_out, double* __restrict__ sd_out, double* __restrict__ quant,
                      double* __restrict__ rhat_out, double* __restrict__ essb_out, double* __restrict__ esst_out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int T = blockDim.x, t = threadIdx.x, G = T / R, r = t / G, lane = t % G;
  const int N = K * S, h = S / 2, M = 2 * K;
  double* red = reinterpret_cast<double*>(smem_raw);  // T
  double* cmb = red + T;                              // R x M
  u64* akey = reinterpret_cast<u64*>(cmb + (size_t)R * M);
  u64* bkey = akey + (size_t)R * N;
  const long long row0 = (long long)blockIdx.x * R;
  const int nr = (int)min((long long)R, n - row0);
  // ---- stage: element e of the tile is (chain e / (S R), sample (e / R) % S, row e % R); rows past n hold zeros
  const long long tot = (long long)N * R;
  for (long long e = t; e < tot; e += T) {
    const int c = (int)(e / ((long long)S * R)), s = (int)((e / R) % S), rr = (int)(e % R);
    const double v = rr < nr ? src[c][(long long)s * n + row0 + rr] : 0.0;
    const u64 k = summary_key(v == 0.0 ? 0.0 : v);  // -0 as +0: ranks treat them as a tie, as numpy compares them
    akey[(size_t)rr * N + (size_t)c * S + s] = k;
    bkey[(size_t)rr * N + (size_t)c * S + s] = k;
  }
  __syncthreads();
  ChainsRow row{akey + (size_t)r * N, bkey + (size_t)r * N, cmb + (size_t)r * M, K, S, h, N};
  // ---- pooled mean and sd (two passes in sample order)
  double acc = 0.0;
  for (int j = lane; j < N; j += G) acc += summary_val(row.a[j]);
  const double mean = summary_group_sum(acc, red, G) / N;
  acc = 0.0;
  for (int j = lane; j < N; j += G) { const double d = summary_val(row.a[j]) - mean; acc += d * d; }
  const double ss = summary_group_sum(acc, red, G);
  summary_sort_rows(bkey, R, N);
  for (int e = t; e < R * np; e += T) {
    const int rr = e / np, jp = e % np;
    if (rr < nr) quant[row0 + rr + (long long)jp * n] = summary_quantile(bkey + (size_t)rr * N, N, probs[jp]);
  }
  const bool live = r < nr;
  double rhat = __longlong_as_double(0x7ff8000000000000LL), essb = rhat, esst = rhat;
  if (h >= 2) {
    double mv, vm;
    // ---- tail-ESS: split indicators of x <= q05 and x <= q95 (pooled quantiles, all K S draws)
    double e2[2];
    for (int j = 0; j < 2; j++) {
      const double q = summary_quantile(row.b, N, j ? 0.95 : 0.05);
      auto ind = [&](int c, int i) { return summary_val(row.a[row.pos(c, i)]) <= q ? 1.0 : 0.0; };
      chains_moments(row, ind, G, lane, red, mv, vm);
      e2[j] = chains_ess(row, ind, G, lane, red, mv, vm, live);
    }
    esst = (isnan(e2[0]) || isnan(e2[1])) ? __longlong_as_double(0x7ff8000000000000LL) : fmin(e2[0], e2[1]);
    // ---- folded R-hat: z-scale of |x - median of the split draws|
    const int Ns = M * h;  // even
    const double med = (row.split_order_stat(Ns / 2 - 1) + row.split_order_stat(Ns / 2)) / 2.0;
    int m0 = 0, m1 = N;
    while (m0 < m1) { const int q = (m0 + m1) >> 1; if (summary_val(row.b[q]) < med) m0 = q + 1; else m1 = q; }
    auto zf = [&](int c, int i) { return row.z_fold(fabs(summary_val(row.a[row.pos(c, i)]) - med), med, m0); };
    chains_moments(row, zf, G, lane, red, mv, vm);
    const double rf = chains_rhat(mv, vm, h);
    // ---- bulk: z-scales in place of the split draws' keys
    double* za = reinterpret_cast<double*>(row.a);
    for (int e = lane; e < Ns; e += G) {
      const int p = row.pos(e / h, e % h);
      za[p] = row.z_bulk(row.a[p]);
    }
    __syncthreads();
    auto zb = [&](int c, int i) { return za[row.pos(c, i)]; };
    chains_moments(row, zb, G, lane, red, mv, vm);
    const double rb = chains_rhat(mv, vm, h);
    rhat = (isnan(rb) || isnan(rf)) ? __longlong_as_double(0x7ff8000000000000LL) : fmax(rb, rf);
    essb = chains_ess(row, zb, G, lane, red, mv, vm, live);
  }
  if (lane == 0 && live) {
    const long long i = row0 + r;
    mean_out[i] = mean;
    sd_out[i] = N > 1 ? sqrt(ss / (N - 1)) : 0.0;
    rhat_out[i] = rhat;
    essb_out[i] = essb;
    esst_out[i] = esst;
  }
}
size_t chains_smem_bytes(int K, int S, int R) {
  return (size_t)kSummaryThreads * sizeof(double) + (size_t)R * 2 * K * sizeof(double) + (size_t)R * 2 * K * S * sizeof(u64);
}
int chains_rows_per_cta(int K, int S, size_t smem_cap) {
  if (K < 1 || S < 1) return 0;
  int R = kSummaryMaxRows;
  while (R >= 1 && chains_smem_bytes(K, S, R) > smem_cap) R >>= 1;
  return R;
}
cudaError_t launch_chains_summary(const double* const* src, long long n, int K, int S, int R, const double* probs, int np, double* mean,
                                  double* sd, double* quant, double* rhat, double* ess_bulk, double* ess_tail, cudaStream_t st) {
  if (n <= 0 || K <= 0 || S <= 0) return cudaSuccess;
  static SmemOptIn opt;
  const size_t smem = chains_smem_bytes(K, S, R);
  cudaError_t e = ensure_dynamic_smem(chains_summary_kernel, smem, opt);
  if (e != cudaSuccess) return e;
  chains_summary_kernel<<<(unsigned)((n + R - 1) / R), kSummaryThreads, smem, st>>>(src, n, K, S, R, probs, np, mean, sd, quant, rhat,
                                                                                   ess_bulk, ess_tail);
  return cudaGetLastError();
}

// ------------------------------------------------------------------ model criteria: PSIS-LOO, WAIC and DIC per observation
// (st_fit_criteria / st_fit_criteria_loglik; DESIGN.md §5e)
// the maximum over the G threads of each row group (as summary_group_sum, pairwise in a fixed order; NaN only if all are)
__device__ __forceinline__ double summary_group_max(double v, double* red, int G) {
  const int t = threadIdx.x, lane = t % G;
  red[t] = v;
  __syncthreads();
  for (int s = G >> 1; s > 0; s >>= 1) {
    if (lane < s) red[t] = fmax(red[t], red[t + s]);
    __syncthreads();
  }
  const double total = red[t - lane];
  __syncthreads();
  return total;
}

constexpr int kGpdSlots = 7;  // grid points of the GPD fit per thread: 30 + floor(sqrt(ceil(0.2 N))) <= 105 <= 7 G (G >= 16)

// One CTA per tile of R rows.  Draw g = c S + s of row i: src[c][s n + i], the log-likelihood itself (P.y == NULL) or w, from
// which ll is formed with y, X, beta_g and tausq_g (every row of the tile reads the same beta_g / tausq_g: read-only path).
// The tile is staged once with coalesced loads (consecutive threads, consecutive rows; T is a multiple of R, so thread t
// stages row t % R throughout and sums its w there for the posterior mean), as order-preserving keys of ll, row-major
// (key[r N + g]), then sorted per row (summary_sort_rows): ascending ll is descending lw = min(ll) - ll, so the PSIS tail is
// sorted positions [0, L) and its cutoff position L.  Per row, over G = T / R threads, every reduction in a fixed order:
// lpd, mean and variance of ll; the GPD fit (each thread takes grid points lane + 1 + u G and sums its point's log1p over the
// tail sequentially; x_m and the smoothed weights are formed on the fly from the keys); the truncated, normalised weights and
// elpd_loo.  out: 8 n doubles, [lpd | elpd_loo | p_loo | pareto_k | elpd_waic | p_waic | -2 mean ll | -2 log N(y; plug-in)],
// NaN at unobserved rows.
__global__ void __launch_bounds__(kSummaryThreads, 1)  // (min. one CTA per SM: ptxas otherwise caps it at 64 registers and spills)
fit_criteria_kernel(const double* const* __restrict__ src, long long n, int K, int S, int R, int L, CritParams P, double* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* red = reinterpret_cast<double*>(smem_raw);  // T
  u64* key = reinterpret_cast<u64*>(red + blockDim.x);  // R x N
  const int T = blockDim.x, t = threadIdx.x, G = T / R, r = t / G, lane = t % G;
  const int N = K * S;
  const double kNaN = __longlong_as_double(0x7ff8000000000000LL), kInf = __longlong_as_double(0x7ff0000000000000LL);
  const double k2pi = 6.283185307179586;  // 2 pi
  const bool par = P.y != nullptr;
  const long long row0 = (long long)blockIdx.x * R;
  const int nr = (int)min((long long)R, n - row0);
  auto observed = [&](int rr) { return rr < nr && (par ? isfinite(P.y[row0 + rr]) : !isnan(src[0][row0 + rr])); };
  // ---- stage: element e of the tile is (draw e / R, row e % R); unobserved rows and rows past n hold zeros
  {
    const int rs = t % R;
    const long long is = row0 + rs;
    const bool live = observed(rs);
    const int js = live && par ? P.mvq[is] : 0;
    const double yv = live && par ? P.y[is] : 0.0;
    double wsum = 0.0;
    for (int g = t / R; g < N; g += G) {
      double ll = 0.0;
      if (live) {
        const int c = g / S, s = g - c * S;
        const double v = src[c][(long long)s * n + is];
        if (par) {
          const double* b = P.beta + ((size_t)g * P.q + js) * P.p;
          double xb = 0.0;
          for (int a = 0; a < P.p; a++) xb += P.X[is + (long long)a * n] * __ldg(b + a);
          const double tau = __ldg(P.tausq + (size_t)g * P.q + js);
          const double res = yv - xb - v;
          ll = -0.5 * log(k2pi * tau) - res * res / (2.0 * tau);
          wsum += v;
        } else {
          ll = v;
        }
      }
      key[(size_t)rs * N + g] = summary_key(ll);
    }
    red[t] = wsum;  // thread t's part of row t % R: draws g = t / R (mod G)
  }
  __syncthreads();
  const double wpart = red[r + R * lane];
  __syncthreads();
  const double wbar = summary_group_sum(wpart, red, G) / N;
  summary_sort_rows(key, R, N);
  const u64* kr = key + (size_t)r * N;
  auto llv = [&](int s) { return summary_val(kr[s]); };
  const double lmin = llv(0), lmax = llv(N - 1);
  // ---- lpd, mean and variance of ll
  double acc = 0.0;
  for (int s = lane; s < N; s += G) acc += exp(llv(s) - lmax);
  const double lpd = lmax + log(summary_group_sum(acc, red, G)) - log((double)N);
  acc = 0.0;
  for (int s = lane; s < N; s += G) acc += llv(s);
  const double mean = summary_group_sum(acc, red, G) / N;
  acc = 0.0;
  for (int s = lane; s < N; s += G) { const double d = llv(s) - mean; acc += d * d; }
  const double ss = summary_group_sum(acc, red, G);
  const double p_waic = N > 1 ? ss / (N - 1) : kNaN;
  // ---- PSIS: the GPD fit of the tail (L is the same for every row: the branch and its barriers are uniform)
  double khat = kInf, sig = 0.0, ec = 0.0;
  if (L >= 5) {
    ec = exp(lmin - llv(L));  // exp(cutoff)
    const bool flat = fabs((lmin - llv(0)) - (lmin - llv(L - 1))) < 2.220446049250313e-16 / 100.0;
    auto xt = [&](int m) { return exp(lmin - llv(L - 1 - m)) - ec; };  // x_m, ascending in m
    const int Mg = 30 + (int)floor(sqrt((double)L));
    const double xstar = xt((int)floor(L / 4.0 + 0.5) - 1), xmax = xt(L - 1);
    double lj[kGpdSlots], thj[kGpdSlots], lm = -kInf;
#pragma unroll
    for (int u = 0; u < kGpdSlots; u++) {
      const int j = lane + 1 + u * G;
      lj[u] = -kInf;
      thj[u] = 0.0;
      if (j <= Mg) {
        const double th = 1.0 / xmax + (1.0 - sqrt((double)Mg / (j - 0.5))) / 3.0 / xstar;
        const double a = -th;
        double ks = 0.0;
        for (int m = 0; m < L; m++) ks += log1p(a * xt(m));
        const double k = ks / L;
        lj[u] = L * (log(a / k) - k - 1.0);
        thj[u] = th;
        lm = fmax(lm, lj[u]);
      }
    }
    const double gm = summary_group_max(lm, red, G);
    double se = 0.0, st = 0.0;
#pragma unroll
    for (int u = 0; u < kGpdSlots; u++)
      if (lane + 1 + u * G <= Mg) { const double e = exp(lj[u] - gm); se += e; st += thj[u] * e; }
    const double sum_e = summary_group_sum(se, red, G);
    const double that = summary_group_sum(st, red, G) / sum_e;
    acc = 0.0;
    for (int m = lane; m < L; m += G) acc += log1p(-that * xt(m));
    const double k = summary_group_sum(acc, red, G) / L;
    sig = -k / that;
    const double kw = (L * k + 5.0) / (L + 10.0);
    khat = flat || isnan(kw) ? kInf : kw;
  }
  const bool smooth = isfinite(khat);
  // ---- the smoothed (tail of a finite k-hat), truncated log weights by sorted position, then their normalisation and elpd_loo
  auto lwv = [&](int s) {
    double v = lmin - llv(s);
    if (smooth && s < L) {
      const double pm = ((L - 1 - s) + 0.5) / L;
      v = log(sig * expm1(-khat * log1p(-pm)) / khat + ec);
    }
    return v > 0.0 ? 0.0 : v;
  };
  double mx = -kInf;
  for (int s = lane; s < N; s += G) mx = fmax(mx, lwv(s));
  mx = summary_group_max(mx, red, G);
  acc = 0.0;
  for (int s = lane; s < N; s += G) acc += exp(lwv(s) - mx);
  const double lsw = mx + log(summary_group_sum(acc, red, G));
  mx = -kInf;
  for (int s = lane; s < N; s += G) mx = fmax(mx, (lwv(s) - lsw) + llv(s));
  mx = summary_group_max(mx, red, G);
  acc = 0.0;
  for (int s = lane; s < N; s += G) acc += exp((lwv(s) - lsw) + llv(s) - mx);
  const double elpd = mx + log(summary_group_sum(acc, red, G));
  if (lane == 0 && r < nr) {
    const long long i = row0 + r;
    const bool live = observed(r);
    double dhat = kNaN;
    if (live && par) {
      const int j = P.mvq[i];
      double mu = 0.0;
      for (int a = 0; a < P.p; a++) mu += P.X[i + (long long)a * n] * P.bbar[j * P.p + a];
      mu += wbar;
      const double tb = P.tbar[j], res = P.y[i] - mu;
      dhat = -2.0 * (-0.5 * log(k2pi * tb) - res * res / (2.0 * tb));
    }
    const double v[8] = {lpd, elpd, lpd - elpd, khat, lpd - p_waic, p_waic, -2.0 * mean, dhat};
#pragma unroll
    for (int c = 0; c < 8; c++) out[(long long)c * n + i] = live ? v[c] : kNaN;
  }
}
int criteria_tail_len(int N, double r_eff) { return (int)ceil(fmin(0.2 * N, 3.0 * sqrt(N / r_eff))); }
cudaError_t launch_fit_criteria(const double* const* src, long long n, int K, int S, int R, double r_eff, const CritParams& P, double* out,
                                cudaStream_t st) {
  if (n <= 0 || K <= 0 || S <= 0) return cudaSuccess;
  const int N = K * S, L = criteria_tail_len(N, r_eff);
  if (L >= 5 && 30 + (int)floor(sqrt((double)L)) > kGpdSlots * (kSummaryThreads / R)) return cudaErrorInvalidValue;
  static SmemOptIn opt;
  const size_t smem = summary_smem_bytes(N, R);
  cudaError_t e = ensure_dynamic_smem(fit_criteria_kernel, smem, opt);
  if (e != cudaSuccess) return e;
  fit_criteria_kernel<<<(unsigned)((n + R - 1) / R), kSummaryThreads, smem, st>>>(src, n, K, S, R, L, P, out);
  return cudaGetLastError();
}

}  // namespace st
