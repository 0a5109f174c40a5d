"""Integrated PSIS-LOO on the GPU (ST_KEEP_LOGLIK_INT, st_get_loglik_int, st_copy_store, st_fit_criteria_integrated,
spamtree(loo_integrated=True); DESIGN.md §5f): the integrated log-likelihood of one sweep against tests/iloo_ref.py on the
sweep's own probes and on dense_twin.Twin's sweep, chains bit for bit the chains without it, the store read in place, the
exact leave-one-out predictive of a model with theta, beta and tausq held fixed, refusals and the entry point."""
import math

import numpy as np
import pytest

import common
import iloo_ref
import launch_configs as lc
import spamtree_b200 as sb
from dense_twin import Twin
from spamtree_b200 import _lib, partition, synth

pytestmark = pytest.mark.gpu

# (the two-level trees of tests/test_iloo_ref.py put every leaf row into one block, wider than a BUILD work group takes)
PROBLEMS = {
    "limited_q1": lambda: common.make_problem(1, 400, limited=True),
    "limited_q2": lambda: common.make_problem(2, 500, limited=True),
    "full_q1": lambda: common.make_problem(1, 625),
    "full_q3": lambda: common.make_problem(3, 900),
    "shape_ref_m_edges": lambda: lc.problem("shape_ref_m_edges"),   # reference blocks at m = 32 / 33 and up to 118
    "q2_n2500_cell36_limited": lambda: lc.problem("q2_n2500_cell36_limited"),  # reference blocks of m = 36 (m > 32)
}
# the Gibbs launches differ between the planner's configurations only in programmatic dependent launch (launch_configs.py)
SWEEP_ROWS = [(p, "default") for p in PROBLEMS] + [(p, "pdl0") for p in ("limited_q2", "full_q3", "shape_ref_m_edges")]


def _keep_loglik_int(m):
    m._chk(_lib.lib.st_keep_samples_on_device(m._h, _lib.ST_KEEP_LOGLIK_INT))


def _near(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1.0)))


@pytest.mark.parametrize("name,config", SWEEP_ROWS, ids=[f"{p}-{c}" for p, c in SWEEP_ROWS])
def test_one_sweep(name, config, monkeypatch):
    pb = PROBLEMS[name]()
    with monkeypatch.context() as mp:
        for k, v in lc.CONFIGS[config]["env"].items():
            mp.setenv(k, v)
        m = common.product_model(pb)
    try:
        n, q = pb["n"], pb["q"]
        y = pb["d"]["y"]
        rng = np.random.default_rng(5)
        tau = np.array([3.0, 5.0, 8.0, 4.0, 6.0])[:q]
        w0 = rng.standard_normal(n) * .5
        m.w = w0
        m.set_tausq_inv(tau)
        assert m.get_loglik_comps_w(0)[0]
        with pytest.raises(sb.SpamTreeError) as ex:
            m.loglik_int()
        assert ex.value.code == 1
        _keep_loglik_int(m)
        z = rng.standard_normal(n)
        m.deal_with_w(z)
        got = m.loglik_int()
        w1 = m.w
        tq = tau[pb["d"]["mv_id"] - 1]
        resid = np.where(np.isfinite(y), y, 0.0) - m.params()["XB"]
        tw = Twin(pb)
        assert np.all(np.isnan(got[~np.isfinite(y)])) and np.all(np.isfinite(got[np.isfinite(y)]))
        # the kernel's formula on the sweep's own Sigi_tot / Smu_tot probes
        worst, nref, nnon = 0.0, 0, 0
        for u in range(tw.nb):
            if tw.obs[u] == 0:
                continue
            ru = tw.rows[u]
            Sig, Smu = m.node_state("Sigi_tot", u), m.node_state("Smu_tot", u)
            if tw.isref[u]:
                Sig = Sig.reshape(ru.size, ru.size)
                nref += 1
            else:
                nnon += 1
            ref = iloo_ref.block_terms(Sig, Smu, w1[ru], z[ru], tq[ru], resid[ru])
            worst = max(worst, _near(got[ru], ref))
        assert nref and nnon
        assert worst <= 1e-10, worst
        # dense_twin's sweep from the same state: its probes, and (two-level and limited trees) the dense prior conditional
        if n <= 1000:
            w_tw, probes = tw.gibbs_sweep(w0, z, tq, resid)
            obs = np.concatenate([tw.rows[u] for u in range(tw.nb) if tw.obs[u] > 0])
            assert common.relerr(w1[obs], w_tw[obs]) < 1e-9
            rows, a, b = iloo_ref.sweep_terms(tw, w0, w_tw, z, tq, resid, probes)
            assert _near(got[rows], a) <= 1e-8
            if name.startswith("limited"):
                assert _near(got[rows], b) <= 1e-8
        # a sweep without the bit leaves the last values alone; the sweep's w does not depend on it
        m2 = common.product_model(pb)
        try:
            m2.w = w0
            m2.set_tausq_inv(tau)
            assert m2.get_loglik_comps_w(0)[0]
            m2.deal_with_w(z)
            assert np.array_equal(m2.w, w1)
        finally:
            m2.close()
    finally:
        m.close()


def _mcmc(m, pb, keep, seed, burn=3, thin=2, **kw):
    npar = pb["theta"].size
    return m.mcmc(synth.default_bounds(pb["q"]), np.eye(npar) * .1, keep, burn, thin, adapting=True, rng_mode=1, seed=seed, **kw)


@pytest.mark.parametrize("q,n,limited", [(1, 625, False), (3, 1500, True)])
def test_chains_unchanged(q, n, limited):
    pb = common.make_problem(q, n, limited=limited)
    a, b = common.product_model(pb), common.product_model(pb)
    try:
        ra = _mcmc(a, pb, 30, seed=7, device_samples=("w",))
        rb = _mcmc(b, pb, 30, seed=7, device_samples=("w", "loglik_int"))
        for key in ("theta_mcmc", "beta_mcmc", "tausq_mcmc", "paramsd", "w_mcmc", "yhat_mcmc", "n_accepted", "n_chol_fail"):
            assert np.array_equal(ra[key], rb[key]), key
        assert np.array_equal(a.stored_draws("w"), b.stored_draws("w"))
        ll = b.stored_draws("loglik_int")
        assert ll.shape == (30, n)
        assert np.array_equal(ll[-1], b.loglik_int(), equal_nan=True)  # the last saved sweep's values
        obs = np.isfinite(pb["d"]["y"])
        assert np.all(np.isnan(ll[:, ~obs])) and np.all(np.isfinite(ll[:, obs]))
    finally:
        a.close()
        b.close()


def test_store_read_in_place():
    pb = common.make_problem(3, 1500, proportions=(.6, .3, .1))
    m = common.product_model(pb)
    try:
        _mcmc(m, pb, 200, seed=4, device_samples=("w", "loglik_int"))
        s0, ll0 = m.summarize("w"), m.stored_draws("loglik_int")
        a = m.fit_criteria(integrated=True)
        b = sb.fit_criteria_loglik(ll0)
        assert set(a) == set(b)
        for k in a:
            assert np.array_equal(a[k], b[k], equal_nan=True), k
        assert math.isnan(a["dic"]) and a["n_obs"] == int(np.isfinite(pb["d"]["y"]).sum())
        again = m.fit_criteria(integrated=True)
        assert all(np.array_equal(a[k], again[k], equal_nan=True) for k in a)
        s1, ll1 = m.summarize("w"), m.stored_draws("loglik_int")
        assert all(np.array_equal(s0[k], s1[k], equal_nan=True) for k in s0)
        assert np.array_equal(ll0, ll1, equal_nan=True)
        cond = m.fit_criteria()  # the conditional criteria of the same run are unaffected
        assert cond["n_samples"] == 200 and np.isfinite(cond["dic"])
        print(f"q = 3, n = 1500, 200 draws: n_k_high {a['n_k_high']} (integrated) against {cond['n_k_high']} (conditional) "
              f"of {a['n_obs']}")
    finally:
        m.close()


def _mc_se(r):
    """batch-means standard error of the mean over axis 0 (draws), b = floor(sqrt(S)) draws per batch"""
    S = r.shape[0]
    bsz = int(math.isqrt(S))
    nb = S // bsz
    bm = r[:nb * bsz].reshape(nb, bsz, *r.shape[1:]).mean(axis=1)
    return bm.std(axis=0, ddof=1) / math.sqrt(nb)


def test_exact_at_fixed_parameters():
    """theta, beta and tausq fixed on a limited tree: every message is current, the sweep's integrated terms are exact
    draws, and elpd_loo must match the closed-form leave-one-out predictive within the Monte Carlo error of the draws"""
    pb = common.make_problem(1, 300, limited=True)
    pb["beta"] = np.array([-1.0, .5, 1.0])
    pb["tausq"] = 0.004  # below the data's noise variance (0.1): w_i follows y_i closely and the conditional k-hat is high
    m = common.product_model(pb)
    try:
        _mcmc(m, pb, 4000, seed=12, burn=200, thin=1, sample_theta=False, sample_beta=False, sample_tausq=False,
              device_samples=("w", "loglik_int"), save_w=False, save_yhat=False)
        got, cond = m.fit_criteria(integrated=True), m.fit_criteria()
        ll = m.stored_draws("loglik_int")
    finally:
        m.close()
    d = pb["d"]
    tw = Twin(pb)
    Q, _ = tw.precision()
    B = np.concatenate([tw.rows[u] for u in range(tw.nb) if tw.obs[u] > 0])
    pos = np.flatnonzero(np.isfinite(d["y"][B]))
    _, _, exact = iloo_ref.exact_loo(Q[np.ix_(B, B)], pos, d["y"][B], (d["X"] @ pb["beta"])[B], np.full(B.size, pb["tausq"]))
    rows = B[pos]
    # Monte Carlo error of the importance-sampling estimate -log mean_s exp(-ll_s) (delta method, batch means over the
    # draws): per row se(mean r) / mean r with r_s = exp(-ll_s); for the total, of sum_i r_is / mean(r_i)
    L = ll[:, rows]
    r = np.exp(-(L - L.min(axis=0)))
    rbar = r.mean(axis=0)
    se_row = _mc_se(r) / rbar
    k = got["pareto_k"][rows]
    ok = k <= got["k_threshold"]
    se_tot = float(_mc_se((r[:, ok] / rbar[ok]).sum(axis=1)))
    assert ok.mean() > 0.95, (ok.sum(), rows.size)
    dev = got["elpd_loo"][rows] - exact
    assert np.all(np.abs(dev[ok]) <= 5 * se_row[ok]), np.max(np.abs(dev[ok]) / se_row[ok])
    assert abs(dev[ok].sum()) <= 5 * se_tot, (dev[ok].sum(), se_tot)
    assert got["n_k_high"] < cond["n_k_high"]
    print(f"fixed parameters, n_obs {rows.size}, 4000 draws: elpd_loo {got['elpd_loo_total']:.3f} against exact {exact.sum():.3f} "
          f"(MC se {se_tot:.3f}); n_k_high {got['n_k_high']} (integrated) against {cond['n_k_high']} (conditional); "
          f"k-hat > 0.5: {np.mean(k > .5):.3f} against {np.mean(cond['pareto_k'][rows] > .5):.3f}")


def test_refusals_leave_the_handle_usable():
    pb = common.make_problem(1, 625)
    m, other = common.product_model(pb), common.product_model(common.make_problem(1, 625, seed=77))
    try:
        with pytest.raises(sb.SpamTreeError) as ex:  # nothing stored
            m.fit_criteria(integrated=True)
        assert ex.value.code == 1 and "no stored draws of the integrated log-likelihood" in str(ex.value)
        with pytest.raises(sb.SpamTreeError) as ex:
            m.stored_draws("loglik_int")
        assert ex.value.code == 1
        with pytest.raises(sb.SpamTreeError) as ex:  # the host-driven chain
            m.mcmc(synth.default_bounds(1), np.eye(pb["theta"].size) * .1, 5, 2, 1, rng_mode=0, device_samples=("loglik_int",))
        assert ex.value.code == 4
        with pytest.raises(sb.SpamTreeError) as ex:  # no sweep over w
            _mcmc(m, pb, 5, seed=1, sample_w=False, device_samples=("loglik_int",))
        assert ex.value.code == 1 and "sample_w" in str(ex.value)
        with pytest.raises(sb.SpamTreeError) as ex:  # more than the device holds
            _mcmc(m, pb, 40_000_000, seed=1, device_samples=("loglik_int",), save_w=False, save_yhat=False)
        assert ex.value.code == 4 and "bytes" in str(ex.value)
        _mcmc(m, pb, 50, seed=3, device_samples=("w",))  # a w store only
        with pytest.raises(sb.SpamTreeError) as ex:
            m.fit_criteria(integrated=True)
        assert ex.value.code == 1
        _mcmc(m, pb, 50, seed=3, device_samples=("loglik_int",))
        first = m.fit_criteria(integrated=True)
        _mcmc(other, common.make_problem(1, 625, seed=77), 50, seed=3, device_samples=("loglik_int",))
        with pytest.raises(sb.SpamTreeError) as ex:  # another data set
            sb.fit_criteria([m, other], integrated=True)
        assert ex.value.code == 1 and "handle 1" in str(ex.value)
        with pytest.raises(sb.SpamTreeError) as ex:
            sb.fit_criteria([], integrated=True)
        assert ex.value.code == 1
        again = m.fit_criteria(integrated=True)
        assert all(np.array_equal(first[k], again[k], equal_nan=True) for k in first)
        for r_eff in (0.0, np.nan):
            with pytest.raises(sb.SpamTreeError) as ex:
                m.fit_criteria(r_eff, integrated=True)
            assert ex.value.code == 1
    finally:
        m.close()
        other.close()
    # a partitioned handle keeps no device store
    t = pb["tree"]
    pl = partition.plan(t, pb["d"]["y"], 2)
    sp = partition.subproblem(pb["d"], t, pl, 0, 2)
    pm = sb.SpamTreeMV(sp["y"], sp["X"], sp["coords"], sp["mv_id"], sp["res_is_ref"], None, None, False, sp["block_names"],
                       sp["block_groups"], None, pb["beta"], pb["theta"], pb["tausq"], csr=sp["csr"],
                       partition=dict(sp, allreduce=lambda ptr, count: None), q=1)
    try:
        with pytest.raises(sb.SpamTreeError) as ex:
            pm._chk(_lib.lib.st_keep_samples_on_device(pm._h, _lib.ST_KEEP_LOGLIK_INT))
        assert ex.value.code == 4
    finally:
        pm.close()


def _same(a, b):
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


@pytest.mark.parametrize("n_chains", [1, 3])
def test_entry_point(n_chains):
    d = synth.make_data(1, 625, missing=0.1, seed=5)
    mc = {"keep": 40, "burn": 5, "thin": 2}
    a = sb.spamtree(d["y"], d["X"], d["coords"], seed=3, mcmc=mc, n_chains=n_chains, fit_criteria=True)
    b = sb.spamtree(d["y"], d["X"], d["coords"], seed=3, mcmc=mc, n_chains=n_chains, fit_criteria=True, loo_integrated=True)
    ci = b.pop("fit_criteria_integrated")
    _same(a, b)
    assert set(ci) == set(b["fit_criteria"])
    assert (ci["n_chains"], ci["n_samples"], ci["n_obs"]) == (n_chains, 40, b["fit_criteria"]["n_obs"])
    assert np.isfinite(ci["elpd_loo_total"]) and math.isnan(ci["dic"])
    cmp = sb.loo_compare(ci, b["fit_criteria"])
    assert cmp["n"] == ci["n_obs"] and np.isfinite(cmp["elpd_diff"])
    only = sb.spamtree(d["y"], d["X"], d["coords"], seed=3, mcmc=mc, n_chains=n_chains, loo_integrated=True)
    _same(only.pop("fit_criteria_integrated"), ci)
    with pytest.raises(sb.SpamTreeError) as ex:
        sb.spamtree(d["y"], d["X"], d["coords"], mcmc=mc, rng_mode=0, loo_integrated=True)
    assert ex.value.code == 1
