"""Model criteria on the GPU (st_fit_criteria, st_fit_criteria_loglik, spamtree(fit_criteria=True)): PSIS-LOO with Pareto
k-hat, WAIC and DIC per observation against the numpy reference of tests/loo_ref.py, stores read in place with no effect
on any handle, pooled chains, refusals, and the detection of a spatial fit against a pure regression."""
import math

import numpy as np
import pytest

import common
import loo_ref
import spamtree_b200 as sb
from spamtree_b200 import synth

pytestmark = pytest.mark.gpu

ROWS = ("lpd", "elpd_loo", "p_loo", "elpd_waic", "p_waic")
TOTALS = ("elpd_loo_total", "se_elpd_loo", "p_loo_total", "looic", "se_looic", "elpd_waic_total", "se_elpd_waic",
          "p_waic_total", "waic", "se_waic", "lpd_total", "dbar", "dhat", "p_dic", "dic", "k_threshold")
COUNTS = ("n_rows", "n_obs", "n_p_waic_high")
LIMIT = 28544  # pooled draws per row one CTA stages (227 KB of shared memory less the reduction scratch)


def _close(a, r, tol=1e-12):
    a, r = np.asarray(a, dtype=np.float64), np.asarray(r, dtype=np.float64)
    if not np.array_equal(np.isnan(a), np.isnan(r)) or not np.array_equal(np.isinf(a), np.isinf(r)):
        return False
    f = np.isfinite(r)
    return bool(np.all(np.abs(a[f] - r[f]) <= np.maximum(tol * np.abs(r[f]), tol)))


def _check(got, ref, dic=True):
    for k in ROWS:
        assert _close(got[k], ref[k]), (k, np.nanmax(np.abs(got[k] - ref[k])))
    assert _close(got["pareto_k"], ref["pareto_k"], 1e-10), np.nanmax(np.abs(got["pareto_k"] - ref["pareto_k"]))
    scale = max(1.0, float(np.nansum(np.abs(ref["lpd"]))) + float(np.nansum(np.abs(ref["p_waic"]))))
    for k in TOTALS:
        if not dic and k in ("dbar", "dhat", "p_dic", "dic"):
            assert math.isnan(got[k]), k
            continue
        a, r = got[k], ref[k]
        assert a == r or (math.isnan(a) and math.isnan(r)) or abs(a - r) <= 1e-12 * max(abs(r), scale), (k, a, r)
    for k in COUNTS:
        assert got[k] == ref[k], (k, got[k], ref[k])
    # n_k_high: rows within 1e-10 of the threshold could go either way; they are set aside and counted
    kr, thr = ref["pareto_k"], ref["k_threshold"]
    near = np.abs(kr - thr) <= 1e-10
    assert near.sum() <= max(1, 0.01 * kr.size)
    gk = got["pareto_k"]
    assert np.sum((gk > thr) & ~near) == np.sum((kr > thr) & ~near)
    assert abs(got["n_k_high"] - ref["n_k_high"]) <= near.sum()


def _synthetic(K, S, n_extra=0, seed=0):
    """(K, S, n) log-likelihoods whose importance ratios exp(-ll) have Pareto tails of shape k (k-hat near k), with a constant
    row, a row with ties, an unobserved row and rows of plain normal ll"""
    rng = np.random.default_rng(seed)
    ks = (0.1, 0.3, 0.45, 0.55, 0.62, 0.68, 0.8, 1.0, 1.5)
    cols = [-0.7 - k * rng.standard_exponential((K, S)) for k in ks]
    cols.append(np.full((K, S), -1.3))                             # constant: k-hat +inf
    cols.append(np.round(-1.0 - 0.4 * rng.standard_exponential((K, S)), 1))  # ties
    cols.append(np.full((K, S), np.nan))                           # unobserved
    cols.append(-0.5 * rng.standard_normal((K, S)) ** 2 - 0.9)
    cols.append(-3.0 * rng.standard_normal((K, S)) ** 2 + 2.0)
    for _ in range(n_extra):
        cols.append(-rng.random() * 2 - rng.random() * rng.standard_exponential((K, S)))
    return np.stack(cols, axis=2)


CASES = [(K, S, 1.0) for K in (1, 2, 4) for S in (1, 2, 5, 17, 20, 21, 1000)] + [(1, 1000, 0.3), (4, 21, 0.3), (2, 5, 0.3)]


@pytest.mark.parametrize("K,S,r_eff", CASES)
def test_loglik_against_numpy(K, S, r_eff):
    ll = _synthetic(K, S, n_extra=20, seed=K * 1000 + S)
    got = sb.fit_criteria_loglik(ll, r_eff)
    ref = loo_ref.criteria(ll, r_eff)
    assert (got["n_chains"], got["n_samples"], got["n_rows"]) == (K, S, ll.shape[2])
    _check(got, ref, dic=False)
    assert math.isnan(got["lpd"][11]) and got["n_obs"] == ll.shape[2] - 1
    if K * S >= 21:
        assert math.isinf(got["pareto_k"][9])  # the constant row
        assert np.all(np.isfinite(got["pareto_k"][:9]))
    else:
        assert np.all(np.isinf(got["pareto_k"][np.arange(ll.shape[2]) != 11]))
    again = sb.fit_criteria_loglik(ll, r_eff)
    assert all(np.array_equal(got[k], again[k], equal_nan=True) for k in got)  # repeated calls are bit-identical


def test_pareto_k_spans_the_ranges():
    ll = _synthetic(4, 1000, seed=3)
    k = sb.fit_criteria_loglik(ll)["pareto_k"]
    assert k[1] < 0.5 and 0.5 < k[3] < 0.7 and k[7] > 0.7 and math.isinf(k[9])


def test_the_draw_limit():
    ll = _synthetic(4, LIMIT // 4, seed=1)[:, :, [0, 5, 9, 11]]  # N at the limit: one row per CTA
    _check(sb.fit_criteria_loglik(ll), loo_ref.criteria(ll), dic=False)
    with pytest.raises(sb.SpamTreeError) as ex:
        sb.fit_criteria_loglik(np.zeros((4, LIMIT // 4 + 1, 2)))
    assert ex.value.code == 4 and str(LIMIT) in str(ex.value)


def test_loglik_refusals():
    ll = _synthetic(2, 30, seed=2)
    for r_eff in (0.0, -1.0, np.nan, np.inf):
        with pytest.raises(sb.SpamTreeError) as ex:
            sb.fit_criteria_loglik(ll, r_eff)
        assert ex.value.code == 1
    for bad in (np.nan, np.inf, -np.inf):
        x = ll.copy()
        x[1, 7, 3] = bad  # one value of an observed row
        with pytest.raises(sb.SpamTreeError) as ex:
            sb.fit_criteria_loglik(x)
        assert ex.value.code == 1
    x = ll.copy()
    x[0, 3, 11] = -1.0  # a number in the NaN row: observed, so its NaNs are refused
    with pytest.raises(sb.SpamTreeError) as ex:
        sb.fit_criteria_loglik(x)
    assert ex.value.code == 1
    for shape in ((0, 5, 3), (2, 0, 3)):
        with pytest.raises(sb.SpamTreeError) as ex:
            sb.fit_criteria_loglik(np.zeros(shape))
        assert ex.value.code == 1
    one = sb.fit_criteria_loglik(ll[0])  # (n_samples, n_rows): one chain
    assert one["n_chains"] == 1 and _close(one["elpd_loo"], loo_ref.criteria(ll[0])["elpd_loo"])


# ---------------------------------------------------------------------------------------------- stores of real runs
def _mcmc(gm, pb, keep, seed, burn=2, thin=1, sd=0.1, **kw):
    npar = pb["theta"].size
    return gm.mcmc(synth.default_bounds(pb["q"]), np.eye(npar) * sd, keep, burn, thin, adapting=True, rng_mode=1, seed=seed, **kw)


def _ref_of_runs(pb, runs, r_eff=1.0):
    """loo_ref on the host arrays of the runs (stacked as chains)"""
    d = pb["d"]
    w = np.concatenate([r["w_mcmc"].T for r in runs])                          # (N, n)
    be = np.concatenate([r["beta_mcmc"].transpose(1, 0, 2) for r in runs])     # (N, p, q)
    ta = np.concatenate([r["tausq_mcmc"].T for r in runs])                     # (N, q)
    ll, dhat = loo_ref.model_loglik(w, be, ta, d["y"], d["X"], d["mv_id"])
    K = len(runs)
    return ll.reshape(K, -1, ll.shape[1]), loo_ref.criteria(ll, r_eff, dhat=dhat)


STORE_CASES = [(1, 625, False, None, 17), (1, 625, False, None, 1000), (3, 1500, False, (.6, .3, .1), 17),
               (3, 1500, True, (.6, .3, .1), 1000), (1, 900, True, None, 1000)]


@pytest.mark.parametrize("q,n,limited,props,keep", STORE_CASES)
def test_store_against_host_arrays(q, n, limited, props, keep):
    pb = common.make_problem(q, n, limited=limited, proportions=props)
    m = common.product_model(pb)
    try:
        run = _mcmc(m, pb, keep, seed=11, device_samples=("w",))
        got = m.fit_criteria()
        ll, ref = _ref_of_runs(pb, [run])
        _check(got, ref)
        assert got["n_obs"] == int(np.sum(np.isfinite(pb["d"]["y"]))) < n  # 10 % missing
        assert all(np.isnan(got["elpd_loo"][~np.isfinite(pb["d"]["y"])]))
        assert _close(sb.fit_criteria_loglik(ll)["elpd_loo"], got["elpd_loo"])
        _check(m.fit_criteria(r_eff=0.3), _ref_of_runs(pb, [run], 0.3)[1])
    finally:
        m.close()


def test_pooled_chains_and_handle_checks():
    pb = common.make_problem(1, 625)
    ms = [common.product_model(pb) for _ in range(3)]
    other = common.make_problem(1, 625, seed=77)  # same size, different data
    mo = common.product_model(other)
    try:
        runs = [_mcmc(m, pb, 200, seed=20 + k, device_samples=("w",)) for k, m in enumerate(ms)]
        got = sb.fit_criteria(ms)
        ll, ref = _ref_of_runs(pb, runs)
        _check(got, ref)
        assert (got["n_chains"], got["n_samples"]) == (3, 200)
        stacked = sb.fit_criteria_loglik(ll)
        for k in ROWS + ("pareto_k",):
            assert _close(got[k], stacked[k], 1e-10 if k == "pareto_k" else 1e-12), k
        _mcmc(mo, other, 200, seed=5, device_samples=("w",))
        with pytest.raises(sb.SpamTreeError) as ex:
            sb.fit_criteria(ms[:2] + [mo])
        assert ex.value.code == 1 and "handle 2" in str(ex.value)
        _mcmc(ms[1], pb, 150, seed=6, device_samples=("w",))  # a different S
        with pytest.raises(sb.SpamTreeError) as ex:
            sb.fit_criteria(ms)
        assert ex.value.code == 1 and "handle 1" in str(ex.value)
    finally:
        for m in ms + [mo]:
            m.close()


def test_deterministic_and_without_side_effects():
    pb = common.make_problem(3, 1500)
    m, twin = common.product_model(pb), common.product_model(pb)
    try:
        for h in (m, twin):
            _mcmc(h, pb, 100, seed=4, device_samples=("w",))
        s0 = m.summarize("w")
        a, b = m.fit_criteria(), m.fit_criteria()
        assert all(np.array_equal(a[k], b[k], equal_nan=True) for k in a)
        s1 = m.summarize("w")
        assert all(np.array_equal(s0[k], s1[k], equal_nan=True) for k in s0)
        ra, rb = _mcmc(m, pb, 20, seed=9, device_samples=("w",)), _mcmc(twin, pb, 20, seed=9, device_samples=("w",))
        for key in ("theta_mcmc", "beta_mcmc", "tausq_mcmc", "paramsd", "w_mcmc", "yhat_mcmc"):
            assert np.array_equal(ra[key], rb[key]), key
    finally:
        m.close()
        twin.close()


def test_refusals_leave_the_handle_usable():
    pb = common.make_problem(1, 625)
    m = common.product_model(pb)
    try:
        with pytest.raises(sb.SpamTreeError) as ex:
            m.fit_criteria()
        assert ex.value.code == 1 and "no stored draws of w" in str(ex.value)
        _mcmc(m, pb, 50, seed=3, device_samples=("yhat",))  # no w store
        with pytest.raises(sb.SpamTreeError) as ex:
            m.fit_criteria()
        assert ex.value.code == 1 and "no stored draws of w" in str(ex.value)
        _mcmc(m, pb, 50, seed=3, device_samples=("w",))
        first = m.fit_criteria()
        for r_eff in (0.0, -1.0, np.nan):
            with pytest.raises(sb.SpamTreeError) as ex:
                m.fit_criteria(r_eff)
            assert ex.value.code == 1
        with pytest.raises(sb.SpamTreeError) as ex:
            sb.fit_criteria([])
        assert ex.value.code == 1
        again = m.fit_criteria()
        assert all(np.array_equal(first[k], again[k], equal_nan=True) for k in first)
    finally:
        m.close()


def test_too_many_stored_draws():
    pb = common.make_problem(1, 625)
    m = common.product_model(pb)
    try:
        _mcmc(m, pb, LIMIT + 1, seed=3, burn=0, device_samples=("w",), save_w=False, save_yhat=False)
        with pytest.raises(sb.SpamTreeError) as ex:
            m.fit_criteria()
        assert ex.value.code == 4 and str(LIMIT) in str(ex.value)
        _mcmc(m, pb, 20, seed=4, device_samples=("w",))  # still usable
        assert m.fit_criteria()["n_samples"] == 20
    finally:
        m.close()


# ---------------------------------------------------------------------------------------------- the entry point
def _same(a, b):
    """a and b bit-identical: dicts and lists item by item, arrays with NaN in the same places (timings skipped)"""
    if isinstance(a, dict):
        assert set(a) == set(b)
        for key in a:
            if key != "mcmc_time":
                _same(a[key], b[key])
    elif isinstance(a, list):
        assert len(a) == len(b)
        for x, y in zip(a, b):
            _same(x, y)
    else:
        assert a is b or np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


def test_entry_point():
    d = synth.make_data(1, 625, missing=0.1, seed=5)
    mc = {"keep": 40, "burn": 5, "thin": 2}
    a = sb.spamtree(d["y"], d["X"], d["coords"], seed=3, mcmc=mc)
    b = sb.spamtree(d["y"], d["X"], d["coords"], seed=3, mcmc=mc, fit_criteria=True)
    crit = b.pop("fit_criteria")
    _same(a, b)
    w, be, ta = b["w_mcmc"].T, b["beta_mcmc"].transpose(1, 0, 2), b["tausq_mcmc"].T
    ll, dhat = loo_ref.model_loglik(w, be, ta, d["y"], d["X"], np.ones(625, np.int64))
    _check(crit, loo_ref.criteria(ll, dhat=dhat))
    # several chains: every chain and summary as without, and the criteria pooled over the chains
    a3 = sb.spamtree(d["y"], d["X"], d["coords"], seed=3, mcmc=mc, n_chains=3)
    b3 = sb.spamtree(d["y"], d["X"], d["coords"], seed=3, mcmc=mc, n_chains=3, fit_criteria=True)
    c3 = b3.pop("fit_criteria")
    _same(a3, b3)
    ch = b3["chains"]
    w = np.concatenate([c["w_mcmc"].T for c in ch])
    be = np.concatenate([c["beta_mcmc"].transpose(1, 0, 2) for c in ch])
    ta = np.concatenate([c["tausq_mcmc"].T for c in ch])
    ll, dhat = loo_ref.model_loglik(w, be, ta, d["y"], d["X"], np.ones(625, np.int64))
    assert c3["n_chains"] == 3
    _check(c3, loo_ref.criteria(ll, dhat=dhat))
    with pytest.raises(sb.SpamTreeError) as ex:
        sb.spamtree(d["y"], d["X"], d["coords"], mcmc=mc, rng_mode=0, fit_criteria=True)
    assert ex.value.code == 1


def test_spatial_fit_beats_a_pure_regression():
    d = synth.make_data(1, 2000, missing=0.1, seed=8)
    mc = {"keep": 300, "burn": 300, "thin": 1}
    sp = sb.spamtree(d["y"], d["X"], d["coords"], seed=2, mcmc=mc, fit_criteria=True)["fit_criteria"]
    rg = sb.spamtree(d["y"], d["X"], d["coords"], seed=2, mcmc=mc, fit_criteria=True,
                     debug={"sample_w": False})["fit_criteria"]
    cmp = sb.loo_compare(sp, rg)
    assert cmp["n"] == sp["n_obs"] == rg["n_obs"]
    assert cmp["elpd_diff"] > 10 * cmp["se_diff"], cmp
    print(f"spatial vs regression: elpd_diff {cmp['elpd_diff']:.1f} (se {cmp['se_diff']:.1f}); n_k_high {sp['n_k_high']} of "
          f"{sp['n_obs']} (spatial), {rg['n_k_high']} (regression); dic {sp['dic']:.1f} vs {rg['dic']:.1f}")
