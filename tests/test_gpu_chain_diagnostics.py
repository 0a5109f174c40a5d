"""Several chains summarised on the GPU (st_summarize_chains, st_summarize_draws, spamtree(n_chains=...)): pooled
quantiles bit for bit against numpy, rank-normalised split-R-hat, bulk-ESS and tail-ESS against the numpy reference of
tests/chain_diag_ref.py, device stores read in place with no effect on any handle, refusals, and the entry point."""
import math

import numpy as np
import pytest

import chain_diag_ref
import common
import spamtree_b200 as sb
from spamtree_b200 import synth

pytestmark = pytest.mark.gpu

PROBS = (0.0, 0.05, 1 / 3, 0.5, 0.975, 1.0)
KEYS = ("mean", "sd", "quantiles", "rhat", "ess_bulk", "ess_tail")
CHAIN_KEYS = ("theta_mcmc", "beta_mcmc", "tausq_mcmc", "paramsd", "w_mcmc", "yhat_mcmc")
LIMIT = 14272  # n_chains x (n_samples + 1) one CTA stages (227 KB of shared memory)


def _same(a, b):
    return all(np.array_equal(a[k], b[k], equal_nan=True) for k in KEYS)


def _check(got, draws, probs):
    """got against the numpy reference on draws (K, S, n)"""
    ref = chain_diag_ref.summarize(draws, probs)
    assert np.array_equal(got["quantiles"], ref["quantiles"]), np.nanmax(np.abs(got["quantiles"] - ref["quantiles"]))
    scale = np.abs(ref["mean"]) + ref["sd"] + 1e-300
    assert np.all(np.abs(got["mean"] - ref["mean"]) <= 1e-13 * scale)
    assert np.all(np.abs(got["sd"] - ref["sd"]) <= 1e-13 * scale)
    for k, tol in (("rhat", 1e-12), ("ess_bulk", 1e-10), ("ess_tail", 1e-10)):
        a, r = got[k], ref[k]
        assert np.array_equal(np.isnan(a), np.isnan(r)), (k, np.flatnonzero(np.isnan(a) != np.isnan(r)))
        fin = np.isfinite(r)
        if k != "rhat":  # a truncation decision a last-bit difference could flip moves the ESS: such rows are counted
            close = ref["margin"] < 1e-12
            assert close.sum() <= 0.01 * close.size, (k, close.sum())
            fin &= ~close
        err = np.abs(a[fin] - r[fin]) / np.abs(r[fin])
        assert np.all(err <= tol), (k, err.max(), np.flatnonzero(fin)[np.argmax(err)])
    return ref


def _ar1(rng, K, S, n, rho):
    x = np.empty((K, S, n))
    x[:, 0] = rng.standard_normal((K, n)) / math.sqrt(1 - rho * rho)
    for s in range(1, S):
        x[:, s] = rho * x[:, s - 1] + rng.standard_normal((K, n))
    return x


def _draws(kind, K, S, n, seed):
    rng = np.random.default_rng(seed)
    if kind == "iid":
        x = rng.standard_normal((K, S, n))
    elif kind == "ar05":
        x = _ar1(rng, K, S, n, 0.5)
    elif kind == "ar95":
        x = _ar1(rng, K, S, n, 0.95)
    elif kind == "shift":
        x = rng.standard_normal((K, S, n)) + rng.random(n) * np.arange(K)[:, None, None]
    elif kind == "scale":
        x = rng.standard_normal((K, S, n)) * (1 + rng.random(n) * np.arange(K)[:, None, None])
    elif kind == "round":
        x = np.round(rng.standard_normal((K, S, n)), 1)
    elif kind == "binary":
        x = (rng.random((K, S, n)) < rng.random(n) * 0.5).astype(np.float64)
    x[:, :, 0] = 2.5  # a constant row: NaN diagnostics
    return x


CASES = ([(kind, K, S) for kind in ("iid", "ar05") for K in (1, 2, 4, 8) for S in (4, 5, 17, 1000)] +
         [("ar95", 4, 1000), ("ar95", 8, 17), ("shift", 4, 1000), ("shift", 8, 17), ("scale", 4, 17), ("scale", 2, 1000),
          ("round", 4, 1000), ("round", 8, 5), ("binary", 4, 1000), ("binary", 2, 17), ("iid", 4, 1), ("iid", 3, 2),
          ("iid", 2, 3)])


@pytest.mark.parametrize("kind,K,S", CASES)
def test_draws_against_numpy(kind, K, S):
    x = _draws(kind, K, S, 37, seed=K * 1000 + S)
    got = sb.summarize_draws(x, PROBS)
    assert (got["n_chains"], got["n_samples"]) == (K, S) and got["quantiles"].shape == (37, len(PROBS))
    assert np.array_equal(got["probs"], np.asarray(PROBS))
    _check(got, x, PROBS)
    assert all(math.isnan(got[k][0]) for k in ("rhat", "ess_bulk", "ess_tail"))  # the constant row
    if S < 4:
        assert np.all(np.isnan(got["rhat"])) and np.all(np.isnan(got["ess_bulk"])) and np.all(np.isnan(got["ess_tail"]))
    assert _same(got, sb.summarize_draws(x, PROBS))  # repeated calls are bit-identical


def test_scalar_draws_and_the_limit():
    x = _draws("ar05", 8, LIMIT // 8 - 1, 3, seed=9)  # K (S + 1) at the limit: one row per CTA
    got = sb.summarize_draws(x, PROBS)
    _check(got, x, PROBS)
    s = sb.summarize_draws(x[:, :, 1], PROBS)  # (n_chains, n_samples): one row
    assert s["mean"].shape == (1,) and all(np.array_equal(s[k][0], got[k][1], equal_nan=True) for k in KEYS)
    with pytest.raises(sb.SpamTreeError) as ex:
        sb.summarize_draws(_draws("iid", 8, LIMIT // 8, 2, seed=1), PROBS)
    assert ex.value.code == 4 and str(LIMIT) in str(ex.value)
    for bad in ((0.5, 1.5), (-0.1,), (np.nan,)):
        with pytest.raises(sb.SpamTreeError) as ex:
            sb.summarize_draws(x, bad)
        assert ex.value.code == 1
    for shape in ((0, 5, 3), (2, 0, 3)):
        with pytest.raises(sb.SpamTreeError) as ex:
            sb.summarize_draws(np.zeros(shape))
        assert ex.value.code == 1


def _mcmc(gm, pb, keep, seed, burn=2, thin=1, sd=0.1, **kw):
    npar = pb["theta"].size
    return gm.mcmc(synth.default_bounds(pb["q"]), np.eye(npar) * sd, keep, burn, thin, adapting=True, rng_mode=1, seed=seed, **kw)


def _same_next_runs(ms, twins, pb, seed):
    for k, (m, t) in enumerate(zip(ms, twins)):
        ra, rb = _mcmc(m, pb, 5, seed + k), _mcmc(t, pb, 5, seed + k)
        for key in CHAIN_KEYS:
            assert np.array_equal(ra[key], rb[key]), (k, key)


@pytest.mark.parametrize("q,n,limited,K", [(1, 625, False, 2), (3, 1500, False, 3), (2, 1200, True, 3)])
def test_stores_read_in_place(q, n, limited, K):
    pb = common.make_problem(q, n, limited=limited)
    ms = [common.product_model(pb, keep_H=False) for _ in range(K)]
    twins = [common.product_model(pb, keep_H=False) for _ in range(K)]
    rs = [_mcmc(m, pb, 41, seed=10 + k, device_samples=("w", "yhat")) for k, m in enumerate(ms)]
    for k, t in enumerate(twins):
        _mcmc(t, pb, 41, seed=10 + k, device_samples=("w", "yhat"))
    for which, key in (("w", "w_mcmc"), ("yhat", "yhat_mcmc")):
        draws = np.stack([r[key].T for r in rs])
        got = sb.summarize_chains(ms, which, PROBS)
        assert (got["n_chains"], got["n_samples"]) == (K, 41)
        assert _same(got, sb.summarize_draws(draws, PROBS))
        assert _same(got, sb.summarize_chains(ms, which, PROBS))
        if which == "w":
            _check(got, draws, PROBS)
    for m, t in zip(ms, twins):  # the stores are as they were
        assert all(np.array_equal(m.summarize("w")[k], t.summarize("w")[k], equal_nan=True) for k in ("mean", "quantiles", "ess"))
    _same_next_runs(ms, twins, pb, seed=50)
    for m in ms + twins:
        m.close()


def test_prediction_stores():
    pb = common.make_problem(1, 625)
    d = pb["d"]
    miss = np.isnan(d["y"])
    cn, xn, mvn = d["coords"][miss], d["X"][miss], d["mv_id"][miss]
    tn = sb.make_tree(d["coords"], d["y"], d["mv_id"], cell_size=25, seed=0, coords_new=cn, mv_id_new=mvn)["new"]
    ms = [common.product_model(pb, keep_H=False) for _ in range(3)]
    prs = []
    for k, m in enumerate(ms):
        _mcmc(m, pb, 20, seed=30 + k, device_samples=("w",))
        prs.append(m.predict_new(cn, xn, mvn, tn, None, seed=5 + k, keep_draws=True))
    for which in ("w_new", "yhat_new"):
        draws = np.stack([p[which].T for p in prs])
        got = sb.summarize_chains(ms, which, PROBS)
        assert got["mean"].size == cn.shape[0]
        assert _same(got, sb.summarize_draws(draws, PROBS))
    for m in ms:
        m.close()


def test_refusals_leave_every_handle_usable():
    pb, pb2 = common.make_problem(1, 625), common.make_problem(1, 700)
    ms = [common.product_model(pb, keep_H=False) for _ in range(3)]
    twins = [common.product_model(pb, keep_H=False) for _ in range(3)]
    other = common.product_model(pb2, keep_H=False)
    host = common.product_model(pb, device=-1)

    def refused(models, code, text, probs=PROBS, which="w"):
        with pytest.raises(sb.SpamTreeError) as ex:
            sb.summarize_chains(models, which, probs)
        assert ex.value.code == code and text in str(ex.value), str(ex.value)

    refused(ms, 1, "handle 0 has no stored draws")  # nothing stored yet
    for k, (m, t) in enumerate(zip(ms, twins)):
        _mcmc(m, pb, 12 if k < 2 else 13, seed=60 + k, device_samples=("w",))
        _mcmc(t, pb, 12 if k < 2 else 13, seed=60 + k, device_samples=("w",))
    _mcmc(other, pb2, 12, seed=1, device_samples=("w",))
    refused(ms, 1, "handle 2 stores 13 draws")         # different S
    refused(ms[:2] + [other], 1, "handle 2 stores")    # different n_rows
    refused(ms[:2], 1, "has no stored draws", which="yhat")
    refused(ms[:2] + [host], 1, "handle 2")            # a host-only handle
    for bad in ((0.5, 1.5), (-0.1,), (np.nan,)):
        refused(ms[:2], 1, "prob", probs=bad)
    before = sb.summarize_chains(ms[:2], "w", PROBS)
    assert _same(before, sb.summarize_chains([ms[0], ms[1]], "w", PROBS))
    _same_next_runs(ms, twins, pb, seed=70)
    for m in ms + twins + [other, host]:
        m.close()


def test_rhat_detects_chains_at_different_theta():
    th = synth.theta_for(1)  # q = 1: sigma^2 = theta[0], phi = theta[3]
    thetas = [th * f for f in ([1, 1, 1, 1], [20, 1, 1, .1], [.02, 1, 1, 20])]
    res = {}
    for label, ths in (("different", thetas), ("same", [th] * 3)):
        ms = []
        for k, t in enumerate(ths):
            pb = common.make_problem(1, 625, theta=t)
            m = common.product_model(pb, keep_H=False)
            m.mcmc(synth.default_bounds(1), np.eye(4) * 0.1, 1000, 200, 1, adapting=True, sample_theta=False, rng_mode=1,
                   seed=80 + k, save_w=False, save_yhat=False, device_samples=("w",))
            ms.append(m)
        res[label] = sb.summarize_chains(ms, "w")["rhat"]
        for m in ms:
            m.close()
    assert np.mean(res["different"] > 1.1) > 0.5, np.quantile(res["different"], (0.1, 0.5, 0.9))
    assert np.mean(res["same"] < 1.05) > 0.95, np.quantile(res["same"], (0.5, 0.9, 0.99))


def test_entry_point_with_several_chains():
    d = synth.make_data(1, 625, missing=0.1, seed=5)
    rng = np.random.default_rng(6)
    cn, xn = rng.random((40, 2)), rng.standard_normal((40, 3))
    kw = dict(mcmc={"keep": 30, "burn": 5, "thin": 2}, coords_new=cn, x_new=xn)
    r = sb.spamtree(d["y"], d["X"], d["coords"], seed=3, n_chains=3, **kw)
    assert set(r) == {"coords", "coordsinfo", "mv_id", "chains", "w_summary", "yhat_summary", "w_new_summary",
                      "yhat_new_summary", "theta_summary", "beta_summary", "tausq_summary"}
    for k in range(3):
        a = sb.spamtree(d["y"], d["X"], d["coords"], seed=3 + k, **kw)
        for key in ("coords", "mv_id"):
            assert np.array_equal(a[key], r[key])
        c = r["chains"][k]
        assert set(c) == set(a) - {"coords", "coordsinfo", "mv_id"}
        for key in c:
            if key == "mcmc_time":
                continue
            va, vb = a[key], c[key]
            if isinstance(va, list):
                assert all(np.array_equal(x, y) for x, y in zip(va, vb)), key
            else:
                assert np.array_equal(np.asarray(va), np.asarray(vb), equal_nan=True), key
    P = (0.025, 0.5, 0.975)
    for which, key in (("w", "w_mcmc"), ("yhat", "yhat_mcmc"), ("w_new", "w_new_mcmc"), ("yhat_new", "yhat_new_mcmc")):
        assert _same(r[which + "_summary"], sb.summarize_draws(np.stack([c[key].T for c in r["chains"]]), P)), which
    th = np.stack([c["theta_mcmc"].T for c in r["chains"]])
    _check(r["theta_summary"], th, P)
    assert r["theta_summary"]["mean"].size == 4
    be = np.stack([c["beta_mcmc"][:, :, 0].T for c in r["chains"]])  # q = 1: p x keep
    assert _same(r["beta_summary"], sb.summarize_draws(be, P))
    # summary_probs: per-chain summaries as a single chain gives them, pooled at the same probs
    r2 = sb.spamtree(d["y"], d["X"], d["coords"], seed=3, n_chains=2, summary_probs=(0.1, 0.9), mcmc=kw["mcmc"])
    a2 = sb.spamtree(d["y"], d["X"], d["coords"], seed=4, summary_probs=(0.1, 0.9), mcmc=kw["mcmc"])
    assert r2["chains"][1]["w_mcmc"] is None
    assert all(np.array_equal(a2["w_summary"][k], r2["chains"][1]["w_summary"][k], equal_nan=True) for k in a2["w_summary"])
    assert np.array_equal(r2["w_summary"]["probs"], [0.1, 0.9])
    # one chain: exactly what the call without n_chains returns
    one, dflt = (sb.spamtree(d["y"], d["X"], d["coords"], seed=3, mcmc=kw["mcmc"], **extra) for extra in ({"n_chains": 1}, {}))
    assert set(one) == set(dflt) and np.array_equal(one["w_mcmc"], dflt["w_mcmc"])
    with pytest.raises(sb.SpamTreeError) as ex:
        sb.spamtree(d["y"], d["X"], d["coords"], n_chains=2, rng_mode=0, mcmc=kw["mcmc"])
    assert ex.value.code == 1


def test_non_finite_draws_are_refused():
    x = _draws("ar05", 4, 17, 12, seed=3)
    for j, v in enumerate((np.nan, np.inf, -np.inf)):
        y = x.copy()
        y[1, 5, 3 + j] = v
        with pytest.raises(sb.SpamTreeError) as ex:
            sb.summarize_draws(y, PROBS)
        assert ex.value.code == 1 and f"draw {1 * 17 * 12 + 5 * 12 + 3 + j} " in str(ex.value)
    _check(sb.summarize_draws(x, PROBS), x, PROBS)


def test_no_handle_to_report_to():
    from spamtree_b200._lib import StChainsSummaryOut, lib
    import ctypes as C
    o = StChainsSummaryOut()
    hs = (C.c_void_p * 1)(None)
    assert lib.st_summarize_chains(hs, 0, 0, None, 0, C.byref(o)) == 1
    assert b"n_chains" in lib.st_last_error(None)
    assert lib.st_summarize_chains(hs, 1, 0, None, 0, C.byref(o)) == 1
    assert b"NULL" in lib.st_last_error(None)
    pb = common.make_problem(1, 625)
    m = common.product_model(pb, keep_H=False)
    _mcmc(m, pb, 8, seed=1, device_samples=("w",))
    closed = common.product_model(pb, keep_H=False)
    closed.close()
    with pytest.raises(sb.SpamTreeError) as ex:  # a closed model first: reported without a handle
        sb.summarize_chains([closed, m], "w")
    assert ex.value.code == 1 and "NULL" in str(ex.value)
    with pytest.raises(sb.SpamTreeError) as ex:
        sb.summarize_chains([m, closed], "w")
    assert ex.value.code == 1 and "handle 1 is NULL" in str(ex.value)
    m.close()


def test_entry_point_parameter_summaries_at_q3():
    d = synth.make_data(3, 1500, proportions=(.5, .3, .2), missing=0.1, seed=7)
    mc = {"keep": 20, "burn": 2, "thin": 1}
    r = sb.spamtree(d["y"], d["X"], d["coords"], d["mv_id"], seed=5, n_chains=2, mcmc=mc,
                    starting=[{"beta": np.zeros(3), "tausq": .1}, {"beta": np.ones(3), "tausq": 1.0}])
    p, q = 3, 3
    P = (0.025, 0.5, 0.975)
    # beta: column a + j p of each sample is beta_mcmc[a, :, j] (p x q, column-major); tausq: row j is tausq_mcmc[j]
    be = np.stack([np.stack([c["beta_mcmc"][a, :, j] for j in range(q) for a in range(p)], axis=1) for c in r["chains"]])
    ta = np.stack([np.stack([c["tausq_mcmc"][j] for j in range(q)], axis=1) for c in r["chains"]])
    assert r["beta_summary"]["mean"].size == p * q and r["tausq_summary"]["mean"].size == q
    assert _same(r["beta_summary"], sb.summarize_draws(be, P))
    assert _same(r["tausq_summary"], sb.summarize_draws(ta, P))
    _check(r["beta_summary"], be, P)
    _check(r["tausq_summary"], ta, P)
    # the second chain is the single-chain call from its own start
    a = sb.spamtree(d["y"], d["X"], d["coords"], d["mv_id"], seed=6, mcmc=mc, starting={"beta": np.ones(3), "tausq": 1.0})
    for key in ("theta_mcmc", "beta_mcmc", "tausq_mcmc", "w_mcmc"):
        assert np.array_equal(a[key], r["chains"][1][key]), key
    for bad in ({"theta": np.ones(15)}, {"w": np.zeros(1500)}):  # starts that would be ignored are refused
        with pytest.raises(sb.SpamTreeError) as ex:
            sb.spamtree(d["y"], d["X"], d["coords"], d["mv_id"], n_chains=2, mcmc=mc, starting=[{}, bad])
        assert ex.value.code == 4
