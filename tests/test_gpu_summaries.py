"""Draws kept on the device and summarised there (st_keep_samples_on_device, st_summarize, st_predict_new_stored):
the store holds what the host arrays receive, the summaries match numpy (quantiles bit for bit), opting in changes nothing
else, prediction from the store equals prediction from host arrays, refusals leave the handle usable, and the
spamtree(..., summary_probs=...) entry point."""
import math

import numpy as np
import pytest

import common
import spamtree_b200 as sb
from spamtree_b200 import synth

pytestmark = pytest.mark.gpu

PROBS = (0.0, 1 / 3, 0.025, 0.5, 0.975, 1.0)
CHAIN_KEYS = ("theta_mcmc", "beta_mcmc", "tausq_mcmc", "paramsd", "w_mcmc", "yhat_mcmc")


def _mcmc(gm, pb, keep, burn=0, thin=1, seed=7, sd=0.1, **kw):
    npar = pb["theta"].size
    return gm.mcmc(synth.default_bounds(pb["q"]), np.eye(npar) * sd, keep, burn, thin, adapting=True, rng_mode=1, seed=seed, **kw)


def _np_summary(x, probs):
    """the definitions of st_summarize restated in numpy; x: rows x S"""
    n, S = x.shape
    out = {"mean": x.mean(axis=1), "sd": x.std(axis=1, ddof=1) if S > 1 else np.zeros(n),
           "quantiles": np.quantile(x, probs, axis=1, method="linear").T}
    b = math.isqrt(S)
    B = S // b
    if S >= 2:
        var = x.var(axis=1, ddof=1)
        sig2 = b * x[:, :B * b].reshape(n, B, b).mean(axis=2).var(axis=1, ddof=1)
        with np.errstate(divide="ignore", invalid="ignore"):
            out["mcse"] = np.where(sig2 > 0, np.sqrt(sig2 / S), np.nan)
            out["ess"] = np.where(sig2 > 0, S * var / sig2, np.nan)
    else:
        out["mcse"] = out["ess"] = np.full(n, np.nan)
    return out


def _check_summary(got, x, probs):
    ref = _np_summary(x, probs)
    assert got["quantiles"].shape == (x.shape[0], len(probs))
    assert np.array_equal(got["quantiles"], ref["quantiles"]), np.max(np.abs(got["quantiles"] - ref["quantiles"]))
    scale = np.abs(ref["mean"]) + ref["sd"] + 1e-300
    assert np.all(np.abs(got["mean"] - ref["mean"]) <= 1e-13 * scale)
    assert np.all(np.abs(got["sd"] - ref["sd"]) <= 1e-13 * scale)
    for k in ("mcse", "ess"):
        a, r = got[k], ref[k]
        assert np.array_equal(np.isnan(a), np.isnan(r)), k
        fin = np.isfinite(r)
        assert np.all(np.abs(a[fin] - r[fin]) <= 1e-12 * np.abs(r[fin])), (k, np.max(np.abs(a[fin] - r[fin]) / np.abs(r[fin])))


def _same(a, b):
    return all(np.array_equal(a[k], b[k], equal_nan=True) for k in ("mean", "sd", "quantiles", "mcse", "ess"))


# (q, n, limited, proportions, keep, burn, thin): S = 17 takes the largest tile (32 rows per CTA), S = 1000 sixteen rows,
# S = 15000 a single row per CTA
CASES = [
    (1, 625, False, None, 17, 0, 1),
    (3, 1500, False, (.6, .3, .1), 4, 3, 2),
    (2, 1200, True, None, 3, 2, 3),
    (1, 625, False, None, 1, 0, 1),
    (1, 625, False, None, 2, 1, 1),
    (1, 625, False, None, 1000, 5, 1),
    (1, 625, False, None, 15000, 0, 1),
]


@pytest.mark.parametrize("q,n,limited,props,keep,burn,thin", CASES)
def test_store_holds_what_the_host_receives(q, n, limited, props, keep, burn, thin):
    pb = common.make_problem(q, n, limited=limited, proportions=props)
    gm = common.product_model(pb, keep_H=False)
    res = _mcmc(gm, pb, keep, burn, thin, device_samples=("w", "yhat"))
    for which, key in (("w", "w_mcmc"), ("yhat", "yhat_mcmc")):
        s = gm.summarize(which, PROBS)
        assert np.array_equal(s["probs"], np.asarray(PROBS))
        _check_summary(s, res[key], PROBS)
        assert _same(s, gm.summarize(which, PROBS))  # repeated calls are bit-identical
    # the same chain with no host arrays at all gives the same summaries, bit for bit
    g2 = common.product_model(pb, keep_H=False)
    r2 = _mcmc(g2, pb, keep, burn, thin, device_samples=("w", "yhat"), save_w=False, save_yhat=False)
    assert r2["w_mcmc"] is None and r2["yhat_mcmc"] is None
    for which in ("w", "yhat"):
        assert _same(gm.summarize(which, PROBS), g2.summarize(which, PROBS)), which
    gm.close()
    g2.close()


def test_opt_in_changes_nothing_else():
    pb = common.make_problem(3, 1500)
    for sd in (0.1, 1e-3, 1e-5, 1e-7):  # the largest proposal scale at which theta moves (15 parameters at q = 3)
        a, b = common.product_model(pb, keep_H=False), common.product_model(pb, keep_H=False)
        ra = _mcmc(a, pb, 12, 4, 2, seed=11, sd=sd)
        rb = _mcmc(b, pb, 12, 4, 2, seed=11, sd=sd, device_samples=("w", "yhat"))
        for k in CHAIN_KEYS:
            assert np.array_equal(ra[k], rb[k]), k
        assert ra["n_accepted"] == rb["n_accepted"]
        if ra["n_accepted"] > 0:
            break
        a.close()
        b.close()
    assert ra["n_accepted"] > 0
    # and again on the same handles (a second run replaces the store; the graphs are reused)
    ra, rb = _mcmc(a, pb, 12, 4, 2, seed=12, sd=sd), _mcmc(b, pb, 12, 4, 2, seed=12, sd=sd, device_samples=("w",))
    for k in CHAIN_KEYS:
        assert np.array_equal(ra[k], rb[k]), k
    with pytest.raises(sb.SpamTreeError) as ex:  # the second run kept w only
        b.summarize("yhat")
    assert ex.value.code == 1
    _check_summary(b.summarize("w", PROBS), rb["w_mcmc"], PROBS)
    a.close()
    b.close()


def _attach(pb, coords_new, mv_new):
    d = pb["d"]
    return sb.make_tree(d["coords"], d["y"], d["mv_id"], cell_size=25, seed=0, coords_new=coords_new, mv_id_new=mv_new,
                        limited_tree=pb["limited"])["new"]


@pytest.mark.parametrize("q,n,limited", [(1, 625, False), (3, 1500, False), (2, 1200, True)])
def test_predict_from_the_store(q, n, limited):
    pb = common.make_problem(q, n, limited=limited)
    d = pb["d"]
    miss = np.isnan(d["y"])
    cn, xn, mvn = d["coords"][miss], d["X"][miss], d["mv_id"][miss]
    tn = _attach(pb, cn, mvn)
    gm = common.product_model(pb, keep_H=False)
    res = _mcmc(gm, pb, 12, 4, 2, seed=7, device_samples=("w",))
    a = gm.predict_new(cn, xn, mvn, tn, None, seed=5, moments=True, keep_draws=True)
    b = gm.predict_new(cn, xn, mvn, tn, res, seed=5, moments=True)
    assert a["n_builds"] == b["n_builds"] >= 1
    for k in ("w_new", "yhat_new", "mean", "sd", "w_new_mean", "w_new_sd", "yhat_new_mean", "yhat_new_sd"):
        assert np.array_equal(a[k], b[k]), k
    for which, key in (("w_new", "w_new"), ("yhat_new", "yhat_new")):
        _check_summary(gm.summarize(which, PROBS), b[key], PROBS)
    # without draws on the host: the same stored draws
    c = gm.predict_new(cn, xn, mvn, tn, None, seed=5, draws=False, keep_draws=True)
    assert "w_new" not in c and np.array_equal(c["w_new_mean"], b["w_new_mean"])
    _check_summary(gm.summarize("w_new", PROBS), b["w_new"], PROBS)
    gm.close()


def _same_next_run(gm, twin, pb, seed):
    """the next normal run of gm equals that of twin, a handle that ran the same successful runs and no refused call (a run
    continues the chain where the handle's last run left it)"""
    ra, rb = _mcmc(gm, pb, 6, 2, 1, seed=seed), _mcmc(twin, pb, 6, 2, 1, seed=seed)
    for k in CHAIN_KEYS:
        assert np.array_equal(ra[k], rb[k]), k
    assert ra["n_accepted"] == rb["n_accepted"]


def test_refusals():
    pb = common.make_problem(1, 625)
    gm, twin = common.product_model(pb, keep_H=False), common.product_model(pb, keep_H=False)
    with pytest.raises(sb.SpamTreeError) as ex:  # nothing stored yet
        gm.summarize("w")
    assert ex.value.code == 1
    with pytest.raises(sb.SpamTreeError) as ex:  # no stored run to predict from
        gm.predict_new(np.zeros((1, 2)), None, None, {"group": np.zeros(1, np.int64), "parents_ptr": np.array([0, 1]),
                                                      "parents_idx": np.zeros(1, np.int64)}, None)
    assert ex.value.code == 1
    with pytest.raises(sb.SpamTreeError) as ex:  # the host-driven chain has no device store
        gm.mcmc(synth.default_bounds(1), np.eye(4) * .1, 3, 0, 1, rng_mode=0, device_samples=("w",))
    assert ex.value.code == 4
    _same_next_run(gm, twin, pb, seed=21)  # (twin is still a fresh handle here)
    _mcmc(gm, pb, 5, device_samples=("w",))
    _mcmc(twin, pb, 5)
    with pytest.raises(sb.SpamTreeError) as ex:  # yhat was not kept
        gm.summarize("yhat")
    assert ex.value.code == 1
    with pytest.raises(sb.SpamTreeError) as ex:  # no stored prediction
        gm.summarize("w_new")
    assert ex.value.code == 1
    for bad in ((0.5, 1.5), (-0.1,), (np.nan,)):
        with pytest.raises(sb.SpamTreeError) as ex:
            gm.summarize("w", bad)
        assert ex.value.code == 1
    assert gm.summarize("w", ())["quantiles"].shape == (625, 0)
    # more draws per row than one CTA stages
    r = _mcmc(gm, pb, 29000, device_samples=("w",), save_w=False, save_yhat=False)
    _mcmc(twin, pb, 29000, save_w=False, save_yhat=False)
    assert r["theta_mcmc"].shape[1] == 29000
    with pytest.raises(sb.SpamTreeError) as ex:
        gm.summarize("w")
    assert ex.value.code == 4 and "28544" in str(ex.value)
    _same_next_run(gm, twin, pb, seed=22)
    gm.close()
    twin.close()

    # a store that cannot fit the device: refused before any iteration, the handle as it was
    pb = common.make_problem(1, 10_000)
    gm, twin = common.product_model(pb, keep_H=False), common.product_model(pb, keep_H=False)

    def too_big():
        with pytest.raises(sb.SpamTreeError) as ex:
            _mcmc(gm, pb, 3_000_000, device_samples=("w", "yhat"), save_w=False, save_yhat=False)
        assert ex.value.code == 4 and "bytes" in str(ex.value)

    too_big()
    _same_next_run(gm, twin, pb, seed=23)  # on a fresh handle
    _mcmc(gm, pb, 4, device_samples=("w",))
    _mcmc(twin, pb, 4)
    before = gm.summarize("w")
    too_big()
    assert _same(before, gm.summarize("w"))  # the last run's store is kept
    _same_next_run(gm, twin, pb, seed=24)
    with pytest.raises(sb.SpamTreeError) as ex:  # (the normal run above replaced the store with none)
        gm.summarize("w")
    assert ex.value.code == 1
    gm.close()
    twin.close()


def test_entry_point():
    d = synth.make_data(1, 625, missing=0.1, seed=5)
    rng = np.random.default_rng(6)
    cn, xn = rng.random((40, 2)), rng.standard_normal((40, 3))
    kw = dict(mcmc={"keep": 30, "burn": 5, "thin": 2}, seed=3, coords_new=cn, x_new=xn)
    probs = (0.05, 0.95)
    a = sb.spamtree(d["y"], d["X"], d["coords"], **kw)
    b = sb.spamtree(d["y"], d["X"], d["coords"], summary_probs=probs, **kw)
    for k in ("w_mcmc", "yhat_mcmc", "w_new_mcmc", "yhat_new_mcmc"):
        assert b[k] is None, k
    for k in a:
        if k in ("mcmc_time", "w_mcmc", "yhat_mcmc", "w_new_mcmc", "yhat_new_mcmc"):
            continue
        va, vb = a[k], b[k]
        if isinstance(va, dict):
            assert all(np.array_equal(va[x], vb[x]) for x in va), k
        elif isinstance(va, list):
            assert all(np.array_equal(x, y) for x, y in zip(va, vb)), k
        else:
            assert np.array_equal(np.asarray(va), np.asarray(vb), equal_nan=True), k
    for k, draws in (("w_summary", "w_mcmc"), ("yhat_summary", "yhat_mcmc"), ("w_new_summary", "w_new_mcmc"),
                     ("yhat_new_summary", "yhat_new_mcmc")):
        assert np.array_equal(b[k]["probs"], np.asarray(probs))
        _check_summary(b[k], a[draws], probs)
    assert set(b) - set(a) == {"w_summary", "yhat_summary", "w_new_summary", "yhat_new_summary"}
