"""The numpy reference of tests/loo_ref.py (PSIS-LOO, WAIC, DIC) pinned on cases checked by hand or from theory; no GPU."""
import math

import numpy as np
import pytest
from scipy import stats

import loo_ref


def test_constant_rows():
    ll = np.full((400, 3), -1.25)
    ll[:, 1] = 0.5
    r = loo_ref.criteria(ll)
    assert np.allclose(r["elpd_loo"], ll[0], rtol=0, atol=1e-14) and np.allclose(r["lpd"], ll[0], rtol=0, atol=1e-14)
    assert np.all(np.abs(r["p_loo"]) <= 1e-14) and np.all(r["p_waic"] == 0)
    assert np.all(np.isinf(r["pareto_k"]))  # a constant tail is left unsmoothed
    assert r["n_k_high"] == 3 and r["n_p_waic_high"] == 0


@pytest.mark.parametrize("N", [1, 2, 5, 20, 21, 22])
def test_short_tails_are_not_smoothed(N):
    ll = np.random.default_rng(N).standard_normal(N) * 2.0
    L = loo_ref.tail_len(N)
    assert (L >= 5) == (N >= 21)
    lw, k = loo_ref.psis(ll)
    if N <= 20:  # plain importance sampling: elpd_loo = -log mean(exp(-ll)) (the harmonic mean)
        assert math.isinf(k)
        elpd = loo_ref.lse(lw + ll)
        assert abs(elpd - (-(loo_ref.lse(-ll) - math.log(N)))) <= 1e-12 * max(1.0, abs(elpd))
    else:
        assert math.isfinite(k)


def test_tail_len_and_r_eff():
    assert loo_ref.tail_len(1000) == 95 and loo_ref.tail_len(4000) == 190 and loo_ref.tail_len(100) == 20
    assert loo_ref.tail_len(1000, 0.3) == 174 and loo_ref.tail_len(21) == 5


def test_quantile_is_scipys_genpareto():
    p = (np.arange(1, 51) - 0.5) / 50
    for k, s in ((0.3, 1.7), (-0.2, 0.5), (0.9, 2.0)):
        assert np.allclose(loo_ref.qgpd(p, k, s), stats.genpareto.ppf(p, c=k, scale=s), rtol=1e-12, atol=0)


@pytest.mark.parametrize("k", [0.2, 0.5, 0.8])
def test_gpdfit_recovers_the_shape(k):
    x = np.sort(stats.genpareto.rvs(c=k, scale=1.3, size=100_000, random_state=np.random.default_rng(int(k * 10))))
    kh, sigma = loo_ref.gpdfit(x)
    assert abs(kh - k) < 0.03, (kh, k)  # sampling sd of the estimate is about (1 + k) / sqrt(n) < 0.006
    assert abs(sigma - 1.3) < 0.05


def _normal_mean(n=40, S=4000, seed=3):
    """y_i ~ N(mu, s2) with s2 known and mu ~ N(0, t2): posterior draws of mu and the exact LOO predictive densities"""
    rng = np.random.default_rng(seed)
    s2, t2 = 1.0, 100.0
    y = rng.standard_normal(n) * math.sqrt(s2) + 0.7
    v = 1.0 / (n / s2 + 1.0 / t2)
    m = v * y.sum() / s2
    mu = m + math.sqrt(v) * rng.standard_normal(S)
    ll = loo_ref.normal_ll(y[None, :], mu[:, None], s2)
    v_i = 1.0 / ((n - 1) / s2 + 1.0 / t2)
    m_i = v_i * (y.sum() - y) / s2
    exact = stats.norm.logpdf(y, m_i, np.sqrt(v_i + s2))
    return y, mu, ll, exact, v, s2


def test_conjugate_normal_mean_loo_is_exact_within_mc_error():
    y, mu, ll, exact, v, s2 = _normal_mean()
    r = loo_ref.criteria(ll)
    assert np.all(r["pareto_k"] < 0.5)
    assert np.all(np.abs(r["elpd_loo"] - exact) < 5e-3), np.max(np.abs(r["elpd_loo"] - exact))
    assert abs(r["elpd_loo_total"] - exact.sum()) < 0.05
    assert abs(r["p_loo_total"] - (r["lpd_total"] - exact.sum())) < 0.05
    assert abs(r["elpd_waic_total"] - exact.sum()) < 0.1  # WAIC is asymptotically LOO


def test_dic_of_a_known_p_d():
    y, mu, ll, exact, v, s2 = _normal_mean()
    dhat = -2.0 * loo_ref.normal_ll(y, mu.mean(), s2)
    r = loo_ref.criteria(ll, dhat=dhat)
    # p_D = n E[(mu - mean mu)^2] / s2: the draws' variance over s2 / n, about 1 (the prior is weak)
    assert abs(r["p_dic"] - y.size * np.var(mu) / s2) < 1e-9
    assert abs(r["p_dic"] - 1.0) < 0.1
    assert abs(r["dic"] - (r["dbar"] + r["p_dic"])) < 1e-9


def test_unobserved_rows_and_totals():
    rng = np.random.default_rng(5)
    ll = rng.standard_normal((2, 50, 6)) * 0.5 - 1.0
    ll[:, :, 2] = np.nan
    r = loo_ref.criteria(ll)
    assert r["n_obs"] == 5 and r["n_rows"] == 6 and all(math.isnan(r[k][2]) for k in ("lpd", "elpd_loo", "pareto_k"))
    obs = np.arange(6) != 2
    assert r["elpd_loo_total"] == pytest.approx(np.sum(r["elpd_loo"][obs]))
    assert r["se_elpd_loo"] == pytest.approx(math.sqrt(5 * np.var(r["elpd_loo"][obs], ddof=1)))
    assert r["looic"] == -2 * r["elpd_loo_total"] and r["k_threshold"] == pytest.approx(0.5)  # N = 100
    assert math.isnan(r["dic"])
    assert loo_ref.criteria(ll[:, :10])["k_threshold"] == pytest.approx(1 - 1 / math.log10(20))  # N = 20: below 0.7
