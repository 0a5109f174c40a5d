"""Rank-normalised split-R-hat, bulk-ESS and tail-ESS (Vehtari, Gelman, Simpson, Carpenter and Buerkner 2021, as ArviZ's
rhat(method="rank") and ess(method="bulk" | "tail") define them) restated in numpy and scipy: the reference the GPU
kernel of st_summarize_chains / st_summarize_draws is checked against (DESIGN.md section 5d).

x is K x S (chains x draws) for one row.  Every function returns NaN where the definitions do; ess() also returns the
smallest |rho_even + rho_odd| its truncation loop decided on (inf when it decided nothing), so that a test can set aside
rows whose truncation point a last-bit difference could move."""
import math

import numpy as np
from scipy import special, stats


def split(x):
    """M = 2K chains of h = S // 2 draws: x[c, :h] and x[c, S - h:] (odd S drops each chain's middle draw)"""
    x = np.asarray(x, dtype=np.float64)
    h = x.shape[1] // 2
    return np.concatenate([x[:, :h], x[:, x.shape[1] - h:]], axis=0) if h else x[:, :0].repeat(2, axis=0)


def z_scale(y):
    """Phi^-1((r - 3/8) / (N + 1/4)) of the average ranks r of all N values, in y's shape"""
    r = stats.rankdata(y.reshape(-1), method="average")
    return special.ndtri((r - 0.375) / (r.size + 0.25)).reshape(y.shape)


def rhat_of(y):
    M, h = y.shape
    B = h * np.var(y.mean(axis=1), ddof=1)
    W = np.mean(np.var(y, axis=1, ddof=1))
    if W == 0:
        return math.nan
    return math.sqrt((B / W + h - 1) / h)


def _acov(y):
    """biased autocovariances of every chain, by direct sums: M x h"""
    M, h = y.shape
    yc = y - y.mean(axis=1, keepdims=True)
    return np.stack([np.correlate(c, c, mode="full")[h - 1:] for c in yc]) / h


def ess_of(y):
    """(ess, margin) of an M x h array"""
    M, h = y.shape
    acov = _acov(y)
    mean_var = np.mean(acov[:, 0]) * h / (h - 1)
    var_plus = mean_var * (h - 1) / h
    if M > 1:
        var_plus += np.var(y.mean(axis=1), ddof=1)
    if var_plus == 0:
        return math.nan, math.inf
    rho = np.zeros(h)
    rho_even, rho_odd = 1.0, 1 - (mean_var - np.mean(acov[:, 1])) / var_plus
    rho[0], rho[1] = rho_even, rho_odd
    margin = abs(rho_even + rho_odd) if 1 < h - 3 else math.inf
    t = 1
    while t < h - 3 and rho_even + rho_odd > 0:
        rho_even = 1 - (mean_var - np.mean(acov[:, t + 1])) / var_plus
        rho_odd = 1 - (mean_var - np.mean(acov[:, t + 2])) / var_plus
        margin = min(margin, abs(rho_even + rho_odd))
        if rho_even + rho_odd >= 0:
            rho[t + 1], rho[t + 2] = rho_even, rho_odd
        t += 2
    max_t = t - 2
    if rho_even > 0:
        rho[max_t + 1] = rho_even
    t = 1
    while t <= max_t - 2:
        if rho[t + 1] + rho[t + 2] > rho[t - 1] + rho[t]:
            rho[t + 1] = rho[t + 2] = (rho[t - 1] + rho[t]) / 2
        t += 2
    tau = -1 + 2 * np.sum(rho[:max_t + 1]) + np.sum(rho[max_t + 1:max_t + 2])
    tau = max(tau, 1 / math.log10(M * h))
    return M * h / tau, margin


def diagnostics(x):
    """dict of rhat, ess_bulk, ess_tail and margin (the smallest of the three ESS loops') of one K x S row"""
    x = np.asarray(x, dtype=np.float64)
    if x.shape[1] // 2 < 2:
        return {"rhat": math.nan, "ess_bulk": math.nan, "ess_tail": math.nan, "margin": math.inf}
    y = split(x)
    zb = z_scale(y)
    zf = z_scale(np.abs(y - np.median(y)))
    rb, rf = rhat_of(zb), rhat_of(zf)
    rhat = math.nan if math.isnan(rb) or math.isnan(rf) else max(rb, rf)
    eb, mb = ess_of(zb)
    q05, q95 = np.quantile(x, (0.05, 0.95), method="linear")
    e05, m05 = ess_of(split((x <= q05).astype(np.float64)))
    e95, m95 = ess_of(split((x <= q95).astype(np.float64)))
    et = math.nan if math.isnan(e05) or math.isnan(e95) else min(e05, e95)
    return {"rhat": rhat, "ess_bulk": eb, "ess_tail": et, "margin": min(mb, m05, m95)}


def summarize(draws, probs):
    """the whole of st_summarize_draws for draws (K, S, n): pooled mean, sd (ddof 1; 0 for one draw), quantiles, and the
    diagnostics of every row, plus its margin"""
    d = np.asarray(draws, dtype=np.float64)
    K, S, n = d.shape
    pooled = d.transpose(2, 0, 1).reshape(n, K * S)
    out = {"mean": pooled.mean(axis=1), "sd": pooled.std(axis=1, ddof=1) if K * S > 1 else np.zeros(n),
           "quantiles": np.quantile(pooled, probs, axis=1, method="linear").T.reshape(n, len(probs))}
    rows = [diagnostics(d[:, :, i]) for i in range(n)]
    for k in ("rhat", "ess_bulk", "ess_tail", "margin"):
        out[k] = np.array([r[k] for r in rows])
    return out
