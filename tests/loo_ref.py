"""PSIS-LOO with Pareto k-hat (R loo 2.x: psis() -> do_psis_i -> psis_smooth_tail -> gpdfit(wip = TRUE, min_grid_pts = 30,
prior 3)), WAIC (loo::waic, p_waic with ddof 1) and DIC at the posterior means (Spiegelhalter et al. 2002, as spBayes' spDiag
uses it) restated in numpy: the reference the GPU kernel of st_fit_criteria / st_fit_criteria_loglik is checked against
(DESIGN.md section 5e).

ll is (N,) for one row: the pooled log-likelihood draws g = c S + s.  Every function follows the definitions literally
(the kernel sorts once and works on sorted positions; ties do not change any output)."""
import math

import numpy as np

DBL_EPS = np.finfo(np.float64).eps


def lse(a):
    a = np.asarray(a, dtype=np.float64)
    m = np.max(a)
    return m + np.log(np.sum(np.exp(a - m)))


def tail_len(N, r_eff=1.0):
    """loo's n_pareto_draws: min(ceil(0.2 N), ceil(3 sqrt(N / r_eff)))"""
    return int(math.ceil(min(0.2 * N, 3.0 * math.sqrt(N / r_eff))))


def gpdfit(x):
    """Zhang and Stephens (2009) as loo's gpdfit(x, wip = TRUE, min_grid_pts = 30), x ascending: (k-hat, sigma)"""
    x = np.asarray(x, dtype=np.float64)
    L = x.size
    M = 30 + int(math.floor(math.sqrt(L)))
    jj = np.arange(1, M + 1, dtype=np.float64)
    xstar = x[int(math.floor(L / 4 + 0.5)) - 1]
    with np.errstate(all="ignore"):
        theta = 1.0 / x[L - 1] + (1.0 - np.sqrt(M / (jj - 0.5))) / 3.0 / xstar
        a = -theta
        k = np.array([np.mean(np.log1p(ai * x)) for ai in a])
        lth = L * (np.log(a / k) - k - 1.0)
        w = np.exp(lth - lse(lth))
        th = np.sum(theta * w)
        kk = np.mean(np.log1p(-th * x))
        sigma = -kk / th
        kh = (L * kk + 5.0) / (L + 10.0)
    return (math.inf if math.isnan(kh) else kh), sigma


def qgpd(p, k, sigma):
    """the GPD quantile loo's qgpd forms: sigma expm1(-k log1p(-p)) / k"""
    return sigma * np.expm1(-k * np.log1p(-p)) / k


def psis(ll, r_eff=1.0):
    """(smoothed, truncated, normalised log weights, k-hat) of one row's ll"""
    ll = np.asarray(ll, dtype=np.float64)
    N = ll.size
    r = -ll
    lw = r - np.max(r)
    L = tail_len(N, r_eff)
    khat = math.inf
    if L >= 5:
        order = np.argsort(lw, kind="stable")
        srt = lw[order]
        tail = srt[N - L:]
        if not abs(np.max(tail) - np.min(tail)) < DBL_EPS / 100:
            cutoff = srt[N - L - 1]
            ec = np.exp(cutoff)
            with np.errstate(all="ignore"):
                khat, sigma = gpdfit(np.exp(tail) - ec)
                if math.isfinite(khat):
                    p = (np.arange(1, L + 1) - 0.5) / L
                    lw[order[N - L:]] = np.log(qgpd(p, khat, sigma) + ec)
    lw = np.where(lw > 0, 0.0, lw)
    return lw - lse(lw), khat


def row(ll, r_eff=1.0):
    """every per-row output for one observed row"""
    ll = np.asarray(ll, dtype=np.float64)
    N = ll.size
    lpd = lse(ll) - math.log(N)
    p_waic = float(np.var(ll, ddof=1)) if N > 1 else math.nan
    lw, khat = psis(ll, r_eff)
    elpd = lse(lw + ll)
    return {"lpd": lpd, "elpd_loo": elpd, "p_loo": lpd - elpd, "pareto_k": khat, "elpd_waic": lpd - p_waic, "p_waic": p_waic,
            "dbar": -2.0 * float(np.mean(ll))}


def normal_ll(y, mu, tausq):
    return -0.5 * np.log(2 * np.pi * tausq) - (y - mu) ** 2 / (2.0 * tausq)


def criteria(ll, r_eff=1.0, dhat=None):
    """ll (K, S, n) or (N, n), NaN rows unobserved; dhat: per-row -2 log N(y; plug-in means) (or None: no DIC)"""
    ll = np.asarray(ll, dtype=np.float64)
    ll = ll.reshape(-1, ll.shape[-1])
    N, n = ll.shape
    keys = ("lpd", "elpd_loo", "p_loo", "pareto_k", "elpd_waic", "p_waic", "dbar")  # (dbar: the per-row -2 mean ll)
    out = {k: np.full(n, np.nan) for k in keys}
    obs = ~np.all(np.isnan(ll), axis=0)
    for i in np.flatnonzero(obs):
        for k, v in row(ll[:, i], r_eff).items():
            out[k][i] = v
    no = int(obs.sum())

    def tot(k):
        return float(np.sum(out[k][obs]))

    def se(k):
        return float(np.sqrt(no * np.var(out[k][obs], ddof=1))) if no > 1 else math.nan
    res = {k: out[k] for k in keys[:-1]}
    with np.errstate(divide="ignore"):  # (N = 1: -inf, as R's loo gives it)
        thr = float(min(1.0 - 1.0 / np.log10(np.float64(N)), 0.7))
    res.update(elpd_loo_total=tot("elpd_loo"), se_elpd_loo=se("elpd_loo"), p_loo_total=tot("p_loo"),
               looic=-2 * tot("elpd_loo"), se_looic=2 * se("elpd_loo"), elpd_waic_total=tot("elpd_waic"),
               se_elpd_waic=se("elpd_waic"), p_waic_total=tot("p_waic"), waic=-2 * tot("elpd_waic"), se_waic=2 * se("elpd_waic"),
               lpd_total=tot("lpd"), k_threshold=thr, n_rows=n, n_obs=no,
               n_k_high=int(np.sum(out["pareto_k"][obs] > thr)), n_p_waic_high=int(np.sum(out["p_waic"][obs] > 0.4)))
    if dhat is None:
        res.update(dbar=math.nan, dhat=math.nan, p_dic=math.nan, dic=math.nan)
    else:
        db, dh = tot("dbar"), float(np.sum(np.asarray(dhat)[obs]))
        res.update(dbar=db, dhat=dh, p_dic=db - dh, dic=db + (db - dh))
    return res


def model_loglik(w, beta, tausq, y, X, mv_id):
    """ll (N, n) of K stacked runs: w (N, n) draws, beta (N, p, q), tausq (N, q), y (n; NaN missing), X (n, p), mv_id 1-based.
    Also the per-row plug-in term -2 log N(y; x' mean(beta[:, j]) + mean(w), mean(tausq_j))."""
    j = np.asarray(mv_id) - 1
    xb = np.einsum("ip,gpi->gi", X, beta[:, :, j])
    ll = normal_ll(y[None, :], xb + w, tausq[:, j])
    ll[:, ~np.isfinite(y)] = np.nan
    mu = np.einsum("ip,pi->i", X, beta.mean(axis=0)[:, j]) + w.mean(axis=0)
    dhat = -2.0 * normal_ll(y, mu, tausq.mean(axis=0)[j])
    return ll, dhat
