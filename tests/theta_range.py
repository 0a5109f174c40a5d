"""The theta box the sampler walks (synth.default_bounds, logit-transformed by par_huvtransf_back) and extended-precision
references for every point of it.  The parity points synth.THETA_Q* sit in a benign corner of that box; a fit starts at the
middle of the box and its Metropolis walk reaches decays near 1e-3 (K nearly singular) and 1e3 (K nearly diagonal, the
exponents of the covariance past the flush of exp_neg), variances of 1e3^2 next to tausq^-1 = 1e3, and the bounds of D, a
and beta.  The references here evaluate the model's formulas in x87 long double (eps ~ 1e-19) and report how close each
block is to losing positive definiteness (the smallest relative Cholesky pivot), which says how much an FP64 algorithm can
be asked for at that point."""
import math
from collections import namedtuple

import numpy as np

from dense_twin import Twin, cov, solve_lower_ld, solve_upper_ld, theta_unpack
from spamtree_b200 import synth

TAU_INV = (10.0, 1e3, 1e-3)  # paired with the points in turn: both ends of the tausq range


def _decays(q):
    """indices of the decay parameters in the theta layout (covariance_functions.cpp:34-92): q = 1 uses thetamv[0]; q = 2
    phi_i and c = thetamv[0]; q >= 3 phi_i and c = thetamv[2]"""
    if q == 1:
        return [3]
    return list(range(2 * q, 3 * q)) + [3 * q + (0 if q == 2 else 2)]


def points(q, n_random=8, seed=20):
    """[(name, theta, tausq_inv)] for q outcomes: the start of spamtree(), the corners of the box that stress the covariance
    and the conditioning, and n_random points drawn uniformly in the logit space of the box (the proposal's space)"""
    import spamtree_b200 as sb
    b = synth.default_bounds(q)
    start = b.mean(axis=1)
    dec = _decays(q)
    out = [("start", start)]

    def at(name, ix, val):
        th = start.copy()
        th[ix] = val
        out.append((name, th))

    at("short", dec, b[dec, 1])        # K nearly diagonal; r h passes the flush of exp_neg
    at("long", dec, 1e-2)
    at("long_min", dec, 1e-3)          # the lower bound: K_pa far from diagonal, small Schur complements
    at("var_hi", list(range(2 * q)), 1e3)   # ai1 = ai2 = 1e3: c1 = ai1^2 = 1e6 on the same-outcome entries
    at("var_lo", list(range(2 * q)), 1e-3)
    npars = 3 * q + (3 if q > 2 else 1)
    if q >= 2:
        at("ai1_neg", [1], -1e3)
        at("D_lo", list(range(npars, b.shape[0])), 1e-3)   # cross-outcome correlation as strong as within-outcome
        at("D_hi", list(range(npars, b.shape[0])), b[npars:, 1])
    if q >= 3:
        at("beta_lo", [3 * q + 1], 1e-3)
        at("beta_hi", [3 * q + 1], 1 - 1e-3)
        at("a_hi", [3 * q], 1e3)
    u = np.random.default_rng(seed + q).uniform(-4, 4, (n_random, b.shape[0]))
    for k in range(n_random):
        out.append((f"random{k}", sb.par_huvtransf_back(u[k], b)))
    return [(name, th, TAU_INV[i % len(TAU_INV)]) for i, (name, th) in enumerate(out)]


def covtab(theta, q):
    """(c1, r1, c2, r2), q x q each, with K(h; i, j) = c1 exp(-r1 h) + c2 exp(-r2 h): make_covtab_hd (st_chain.hpp) in
    float64 by the same operations, so that it is the table the device evaluates bit for bit"""
    th = [float(x) for x in theta]
    ai1, ai2, phi, tm, D = (np.asarray(a, dtype=np.float64) for a in theta_unpack(np.asarray(th), q))
    c1, r1, c2, r2 = (np.zeros((q, q)) for _ in range(4))
    if q == 1:
        c1[0, 0], r1[0, 0] = th[0], th[3]
        return c1, r1, c2, r2
    for i in range(q):
        for j in range(q):
            v = float(D[i, j])
            if q > 2:
                ps = math.exp(0.5 * float(tm[1]) * math.log1p(float(tm[0]) * v))
                psi2, c = ps * ps, float(tm[2])
            else:
                ps, psi2, c = math.sqrt(v + 1), v + 1.0, float(tm[0])
            if v == 0:
                c1[i, j], r1[i, j] = float(ai1[i]) * float(ai1[i]) / psi2, c / ps
                c2[i, j], r2[i, j] = float(ai2[i]) * float(ai2[i]), float(phi[i])
            else:
                c1[i, j], r1[i, j] = float(ai1[i]) * float(ai1[j]) / psi2, c / ps
    return c1, r1, c2, r2


def chol_margin(A, scale=None):
    """lower Cholesky factor of A in long double (dense_twin.chol_ld's algorithm) and its smallest relative pivot
    min_j d_j / scale_j, d_j the pivot before its square root (scale: diag(A)).  (None, margin) if a pivot is not
    positive: A is not positive definite even in extended precision."""
    A = np.array(A, dtype=np.longdouble)
    s = np.diag(A).copy() if scale is None else np.asarray(scale, dtype=np.longdouble)
    n = A.shape[0]
    margin = 1.0
    for j in range(n):
        d = A[j, j] - A[j, :j] @ A[j, :j]
        margin = min(margin, float(d / s[j]))
        if not d > 0:
            return None, margin
        A[j, j] = np.sqrt(d)
        if j + 1 < n:
            A[j + 1:, j] = (A[j + 1:, j] - A[j + 1:, :j] @ A[j, :j]) / A[j, j]
    return np.tril(A), margin


LdBlock = namedtuple("LdBlock", "H Ri margin_pa margin_R cond_pa")


def ld_block(coords, mv, ru, rp, theta, q, isref):
    """dense_twin.block_truth_ld (H = K_{u,pa} K_pa^-1, Ri = chol(R)^-1 or 1 / sqrt(diag R), R = K_uu - H K_{pa,u}) plus
    the smallest relative Cholesky pivot of K_pa and of R, the latter relative to diag(K_uu): the margin by which each is
    positive definite, 1 for a diagonal matrix, <= 0 for one that is not (H and Ri are then None), and cond_2(K_pa)."""
    ld = np.longdouble
    Kuu = cov(coords[ru], mv[ru], coords[ru], mv[ru], theta, q, ld)
    m = ru.size
    if rp.size:
        Kpp = cov(coords[rp], mv[rp], coords[rp], mv[rp], theta, q, ld)
        cond = float(np.linalg.cond(Kpp.astype(np.float64)))
        L, mpa = chol_margin(Kpp)
        if L is None:
            return LdBlock(None, None, mpa, mpa, cond)
        Y = solve_lower_ld(L, cov(coords[rp], mv[rp], coords[ru], mv[ru], theta, q, ld))
        H = solve_upper_ld(L.T, Y).T
        R = Kuu - Y.T @ Y
    else:
        H, R, mpa, cond = np.zeros((m, 0), dtype=ld), Kuu, 1.0, 1.0
    if isref:
        LR, mR = chol_margin(R, np.diag(Kuu))
        Ri = None if LR is None else solve_lower_ld(LR, np.eye(m, dtype=ld))
    else:
        dR = np.diag(R)
        mR = float(np.min(dR / np.diag(Kuu)))
        Ri = 1 / np.sqrt(dR) if mR > 0 else None
    return LdBlock(H, Ri, mpa, mR, cond)


def ld_blocks(pb, theta):
    """(Twin of the problem, {observed block: LdBlock})"""
    tw = Twin(pb, theta)
    out = {}
    for u in range(tw.nb):
        if tw.obs[u]:
            out[u] = ld_block(tw.coords, tw.mv, tw.rows[u], tw.prow(u), theta, tw.q, bool(tw.isref[u]))
    return tw, out


def _blocks(pb, theta, blocks):
    return ld_blocks(pb, theta) if blocks is None else blocks


def ld_loglik(pb, theta, w, blocks=None):
    """(log-density of w, log-determinant) block by block in long double: sum of log diag Ri and of
    -1/2 |Ri (w_u - H w_pa)|^2 over the observed blocks, minus nobs / 2 log(2 pi) (Twin.loglik's quantity without its
    dense float64 Q, which is itself ill-conditioned at the ends of the box).  NaN if a block is not positive definite."""
    tw, bl = _blocks(pb, theta, blocks)
    wl = np.asarray(w, dtype=np.longdouble)
    logdet, quad, nobs = np.longdouble(0), np.longdouble(0), 0
    for u, b in bl.items():
        if b.Ri is None:
            return math.nan, math.nan
        ru, rp = tw.rows[u], tw.prow(u)
        e = wl[ru] - (b.H @ wl[rp] if rp.size else 0)
        if tw.isref[u]:
            logdet += np.sum(np.log(np.diag(b.Ri)))
            r = b.Ri @ e
        else:
            logdet += np.sum(np.log(b.Ri))
            r = b.Ri * e
        quad += r @ r
        nobs += ru.size
    return float(logdet - 0.5 * quad - np.longdouble(0.5 * nobs) * np.log(2 * np.pi, dtype=np.longdouble)), float(logdet)


def ld_gibbs_sweep(pb, theta, w, z, tausq_inv_row, resid, blocks=None):
    """dense_twin.Twin.gibbs_sweep (the reference's message timing) in long double from the long-double blocks: the new w
    and every observed block's (Sigi_tot, Smu_tot)"""
    tw, bl = _blocks(pb, theta, blocks)
    ld = np.longdouble
    w = np.asarray(w, dtype=ld).copy()
    z, tq, resid = (np.asarray(a, dtype=ld) for a in (z, tausq_inv_row, resid))
    msgS = {u: np.zeros((tw.rows[u].size,) * 2, dtype=ld) for u in range(tw.nb)}
    msgM = {u: np.zeros(tw.rows[u].size, dtype=ld) for u in range(tw.nb)}
    probes = {}
    for lev in reversed(tw.levels):
        for u in [u for u in bl if tw.level[u] == lev]:
            ru, rp = tw.rows[u], tw.prow(u)
            H, Ri = bl[u].H, bl[u].Ri
            prec = Ri.T @ Ri if tw.isref[u] else np.diag(Ri ** 2)
            Hw = H @ w[rp] if rp.size else np.zeros(ru.size, dtype=ld)
            if tw.isref[u]:
                Sig = prec + msgS[u] + np.diag(tq[ru])
                Smu = prec @ Hw + msgM[u] + tq[ru] * resid[ru]
                L, _ = chol_margin(Sig)
                w[ru] = solve_upper_ld(L.T, solve_lower_ld(L, Smu) + z[ru])   # L^-T (L^-1 Smu + z)
                probes[u] = (Sig, Smu)
            else:
                sig = np.diag(prec) + tq[ru]
                smu = np.diag(prec) * Hw + tq[ru] * resid[ru]
                w[ru] = smu / sig + z[ru] / np.sqrt(sig)
                probes[u] = (sig, smu)
            off = 0
            for a in tw.parents[u]:
                ma = tw.rows[a].size
                Ha = H[:, off:off + ma]
                others = np.ones(rp.size, dtype=bool)
                others[off:off + ma] = False
                msgS[a] = msgS[a] + Ha.T @ prec @ Ha
                msgM[a] = msgM[a] + Ha.T @ prec @ (w[ru] - H[:, others] @ w[rp][others])
                off += ma
    return w, probes


def ld_dense_precision(pb, theta, blocks=None):
    """Q = sum over observed blocks of (I - H_u)' Ri'Ri (I - H_u) in long double, n x n (Twin.precision's matrix), for
    iloo_ref.dense_terms"""
    tw, bl = _blocks(pb, theta, blocks)
    n = tw.y.size
    Q = np.zeros((n, n), dtype=np.longdouble)
    for u, b in bl.items():
        ru, rp = tw.rows[u], tw.prow(u)
        m = ru.size
        B = np.concatenate([np.eye(m, dtype=np.longdouble), -b.H], axis=1)
        RB = b.Ri @ B if tw.isref[u] else b.Ri[:, None] * B
        cols = np.concatenate([ru, rp])
        Q[np.ix_(cols, cols)] += RB.T @ RB
    return Q


def ld_predict(pb, theta, tree_new, coords_new, mv_new, w, dtype=np.longdouble):
    """conditional mean H w_pa and variance (Schur complement) K_ii - H K_{pa,i} of every new row given its group's parent
    rows (the "new" entry of make_tree(..., coords_new=...)), by Cholesky of K_pa and triangular solves in `dtype` (float64:
    the algorithm an FP64 reference would run).  Returns (mean, var, K_ii, smallest relative pivot of the K_pa)."""
    d, t = pb["d"], pb["tree"]
    q = pb["q"]
    ip, ii = t["indexing_ptr"], t["indexing_idx"]
    grp, pp, pi = tree_new["group"], tree_new["parents_ptr"], tree_new["parents_idx"]
    nn = len(coords_new)
    mean, var, kii = (np.zeros(nn, dtype=dtype) for _ in range(3))
    margin = 1.0
    for g in range(len(pp) - 1):
        sel = np.flatnonzero(grp == g)
        if not sel.size:
            continue
        pa = np.concatenate([ii[ip[b]:ip[b + 1]] for b in pi[pp[g]:pp[g + 1]]])
        Kpp = cov(d["coords"][pa], d["mv_id"][pa], d["coords"][pa], d["mv_id"][pa], theta, q, dtype)
        Kpi = cov(d["coords"][pa], d["mv_id"][pa], coords_new[sel], mv_new[sel], theta, q, dtype)
        k = np.diag(cov(coords_new[sel], mv_new[sel], coords_new[sel], mv_new[sel], theta, q, dtype))
        if dtype == np.longdouble:
            L, mg = chol_margin(Kpp)
            margin = min(margin, mg)
            if L is None:
                mean[sel], var[sel] = np.nan, np.nan
                continue
            Y, x = solve_lower_ld(L, Kpi), solve_lower_ld(L, np.asarray(w, dtype=dtype)[pa])
        else:
            import scipy.linalg as sl
            L = np.linalg.cholesky(Kpp)
            Y, x = sl.solve_triangular(L, Kpi, lower=True), sl.solve_triangular(L, np.asarray(w)[pa], lower=True)
        mean[sel], var[sel], kii[sel] = Y.T @ x, k - np.sum(Y * Y, axis=0), k
    return mean, var, kii, margin
