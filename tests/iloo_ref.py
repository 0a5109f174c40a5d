"""numpy statement of the integrated log-likelihood (DESIGN.md §5f) and of the exact leave-one-out predictive of the Gaussian
model at fixed theta, beta and tausq, for tests/test_iloo_ref.py (CPU) and tests/test_gpu_loo_integrated.py."""
import numpy as np


def norm_logpdf(x, mean, var):
    return -0.5 * (np.log(2 * np.pi * var) + (x - mean) ** 2 / var)


def block_terms(Sig, Smu, w, z, tq, resid):
    """ll_a for every row a of one block of a Gibbs sweep, from what the sweep had when it drew the block: Sigi_tot (m x m; a
    non-reference block: its m scalars), Smu_tot, the block's new w = L^-T (L^-1 Smu + z) with L = chol(Sigi_tot), z,
    tausq_inv and y - XB of its rows.  Sigi_tot w - Smu = L z; taking row a's observation out of both leaves the prior
    conditional of w_a given the rest of w: precision Q'_aa = Sigi_tot_aa - tausq_inv_a, mean w_a - (L z + tq (resid - w))_a / Q'_aa.
    ll_a = log N(resid_a; that mean, 1 / Q'_aa + 1 / tausq_inv_a)."""
    Sig, Smu, w, z, tq, resid = (np.asarray(a, dtype=np.float64) for a in (Sig, Smu, w, z, tq, resid))
    if Sig.ndim == 1:
        Lz, qd = np.sqrt(Sig) * z, Sig - tq
    else:
        Lz, qd = np.linalg.cholesky((Sig + Sig.T) / 2) @ z, np.diag(Sig) - tq
    mean = w - (Lz + tq * (resid - w)) / qd
    return norm_logpdf(resid, mean, 1 / qd + 1 / tq)


def dense_terms(Q, state, rows, tq, resid):
    """the same from the dense prior precision Q of w (n x n) at the state of w the block is drawn from: w_a given the rest
    of w is N(w_a - (Q state)_a / Q_aa, 1 / Q_aa), whatever w_a itself is"""
    qd = np.diag(Q)[rows]
    mean = state[rows] - (Q[rows] @ state) / qd
    return norm_logpdf(resid, mean, 1 / qd + 1 / tq)


def sweep_terms(tw, w_before, w_after, z, tausq_inv_row, resid, probes):
    """both statements for every observed row of a sweep of dense_twin.Twin (probes from Twin.gibbs_sweep): the sweep runs
    the levels deepest first, so block u is drawn with every deeper level (and its own) at w_after, the shallower ones at
    w_before (blocks of one level share no child, so they do not enter each other's conditionals).  Returns
    (rows, from the probes, from the dense precision)."""
    Q, _ = tw.precision()
    rows, a, b = [], [], []
    for u, (Sig, Smu) in probes.items():
        ru = tw.rows[u]
        a.append(block_terms(Sig, Smu, w_after[ru], z[ru], tausq_inv_row[ru], resid[ru]))
        state = np.where(np.isin(np.arange(w_before.size), _rows_at_or_below(tw, tw.level[u])), w_after, w_before)
        b.append(dense_terms(Q, state, ru, tausq_inv_row[ru], resid[ru]))
        rows.append(ru)
    return np.concatenate(rows), np.concatenate(a), np.concatenate(b)


def _rows_at_or_below(tw, lev):
    return np.concatenate([tw.rows[u] for u in range(tw.nb) if tw.obs[u] > 0 and tw.level[u] >= lev])


def exact_loo(Q, rows, y, xb, tausq):
    """the exact leave-one-out predictive of the observed rows `rows` at fixed theta, beta and tausq: y ~ N(xb, Sigma) with
    Sigma = Q^-1 + tausq I over the rows of the observed blocks (Q restricted to them), so y_i given y_-i is
    N(y_i - [Sigma^-1 r]_i / [Sigma^-1]_ii, 1 / [Sigma^-1]_ii), r = y - xb.  Returns (mean, var, log density at y_i);
    tausq: per row."""
    Sig = np.linalg.inv(Q) + np.diag(tausq)
    P = np.linalg.inv(Sig[np.ix_(rows, rows)])
    r = (y - xb)[rows]
    d = np.diag(P)
    mean = y[rows] - (P @ r) / d
    return mean, 1 / d, norm_logpdf(y[rows], mean, 1 / d)


def brute_loo(Q, rows, y, xb, tausq, i):
    """the same for row rows[i] by conditioning the joint normal of the observed rows on the others"""
    Sig = (np.linalg.inv(Q) + np.diag(tausq))[np.ix_(rows, rows)]
    o = np.arange(rows.size) != i
    r = (y - xb)[rows]
    k = Sig[i, o]
    sol = np.linalg.solve(Sig[np.ix_(o, o)], np.stack([r[o], k], axis=1))
    return xb[rows[i]] + k @ sol[:, 0], Sig[i, i] - k @ sol[:, 1]
