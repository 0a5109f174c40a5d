"""Prediction at new locations from saved samples (SpamTreeMV.predict_new, st_predict_new): the same draws as the chain's
own prediction of its NaN rows, the dense conditional mean / sd of numpy, reproducible draws, no side effect on the fitted
handle, and the spamtree(..., coords_new=...) entry point."""
import numpy as np
import pytest

import common
import dense_twin as dt
import philox_host as ph
from common import relerr
import spamtree_b200 as sb
from spamtree_b200 import partition, synth

pytestmark = pytest.mark.gpu


def _mcmc(gm, pb, keep=12, burn=4, thin=2, seed=7, sd=0.1):
    npar = pb["theta"].size
    return gm.mcmc(synth.default_bounds(pb["q"]), np.eye(npar) * sd, keep, burn, thin, adapting=True, rng_mode=1, seed=seed)


def _attach(pb, coords_new, mv_new):
    d = pb["d"]
    return sb.make_tree(d["coords"], d["y"], d["mv_id"], cell_size=25, seed=0, coords_new=coords_new, mv_id_new=mv_new,
                        limited_tree=pb["limited"])["new"]


def _theta_of_prediction(theta_mcmc):
    """the theta the chain's in-chain prediction was built at: need_update of spamtree_fit.cpp:300 replayed"""
    used, pp, out = None, None, np.empty_like(theta_mcmc)
    for s in range(theta_mcmc.shape[1]):
        th = theta_mcmc[:, s]
        if used is None or np.any(np.abs(th - pp) > 1e-5):
            used = th.copy()
        pp = th.copy()
        out[:, s] = used
    return out


@pytest.mark.parametrize("q,n,limited", [(1, 625, False), (3, 1500, False), (2, 1200, True)])
def test_same_draws_as_the_chain(q, n, limited):
    pb = common.make_problem(q, n, limited=limited)
    d = pb["d"]
    miss = np.isnan(d["y"])
    rows = np.flatnonzero(miss)
    keep, burn, thin, seed = 12, 4, 2, 7
    for sd in (0.1, 1e-3, 1e-5, 1e-7):  # the largest proposal scale at which theta moves (15 parameters at q = 3)
        gm = common.product_model(pb, keep_H=False)
        res = _mcmc(gm, pb, keep, burn, thin, seed, sd=sd)
        if res["n_accepted"] > 0:
            break
        gm.close()
    assert res["n_accepted"] > 0
    iters = burn + thin * np.arange(keep)
    z = np.stack([ph.normal(seed, rows.astype(np.uint64), m) for m in iters], axis=1)
    eps = np.stack([ph.normal(seed, rows.astype(np.uint64), ph.K_COUNTER_YHAT + m + 1) for m in iters], axis=1)
    samples = dict(res, theta_mcmc=_theta_of_prediction(res["theta_mcmc"]))
    out = gm.predict_new(d["coords"][miss], d["X"][miss], d["mv_id"][miss], _attach(pb, d["coords"][miss], d["mv_id"][miss]),
                         samples, z=z, eps=eps)
    ew, ey = relerr(out["w_new"], res["w_mcmc"][miss]), relerr(out["yhat_new"], res["yhat_mcmc"][miss])
    print(f"q={q} n={n} limited={limited}: w relerr {ew:.2e}, yhat relerr {ey:.2e}, BUILDs {out['n_builds']}")
    assert ew <= 1e-9 and ey <= 1e-9
    gm.close()


def _dense_truth(pb, tree_new, cn, mvn, w, theta):
    d, t = pb["d"], pb["tree"]
    q = pb["q"]
    ip, ii = t["indexing_ptr"], t["indexing_idx"]
    mean, var = np.zeros(len(cn)), np.zeros(len(cn))
    grp, pp, pi = tree_new["group"], tree_new["parents_ptr"], tree_new["parents_idx"]
    for g in range(len(pp) - 1):
        sel = np.flatnonzero(grp == g)
        pa = np.concatenate([ii[ip[b]:ip[b + 1]] for b in pi[pp[g]:pp[g + 1]]])
        Kpp = dt.cov(d["coords"][pa], d["mv_id"][pa], d["coords"][pa], d["mv_id"][pa], theta, q)
        Kip = dt.cov(cn[sel], mvn[sel], d["coords"][pa], d["mv_id"][pa], theta, q)
        Kii = np.diag(dt.cov(cn[sel], mvn[sel], cn[sel], mvn[sel], theta, q))
        H = np.linalg.solve(Kpp, Kip.T).T
        mean[sel] = H @ w[pa]
        var[sel] = Kii - np.einsum("ij,ij->i", H, Kip)
    return mean, var


@pytest.mark.parametrize("q,limited", [(1, False), (2, False), (3, False), (1, True), (3, True)])
def test_dense_truth(q, limited):
    pb = common.make_problem(q, 1500, limited=limited)
    d = pb["d"]
    rng = np.random.default_rng(11)
    obs_at = d["coords"][np.flatnonzero(np.isfinite(d["y"]))[100]]
    cn = np.vstack([rng.random((300, 2)) * 1.4 - 0.2,                 # inside and outside the unit square
                    obs_at + (rng.random((350, 2)) - .5) * 1e-5,         # a cluster around one parent block (pseudo-block split)
                    obs_at[None, :]])                                    # a point on an observed location
    mvn = rng.integers(1, q + 1, cn.shape[0])
    mvn[-1] = d["mv_id"][np.flatnonzero(np.isfinite(d["y"]))[100]]
    tn = _attach(pb, cn, mvn)
    assert np.bincount(tn["group"]).max() > 300
    gm = common.product_model(pb, keep_H=False)
    w = rng.standard_normal(pb["n"])
    samples = {"theta_mcmc": pb["theta"][:, None], "beta_mcmc": np.zeros((3, 1, q)), "tausq_mcmc": np.full((q, 1), .1),
               "w_mcmc": w[:, None]}
    out = gm.predict_new(cn, None, mvn, tn, samples, moments=True)
    mean, var = _dense_truth(pb, tn, cn, mvn, w, pb["theta"])
    em = relerr(out["mean"][:, 0], mean)
    ev = np.max(np.abs(out["sd"][:, 0] ** 2 - var)) / np.max(np.abs(var))
    print(f"q={q} limited={limited}: mean relerr {em:.2e}, var relerr {ev:.2e}, groups {tn['n_groups']}")
    assert em <= 1e-9 and ev <= 1e-9
    assert np.all(np.isfinite(out["sd"])) and np.all(out["sd"] >= 0) and np.all(np.isfinite(out["mean"]))
    gm.close()


def test_reproducible_and_deterministic():
    pb = common.make_problem(2, 1200)
    d = pb["d"]
    gm = common.product_model(pb, keep_H=False)
    res = _mcmc(gm, pb, keep=10, burn=2, thin=1)
    rng = np.random.default_rng(5)
    cn = rng.random((500, 2))
    mvn = rng.integers(1, 3, 500)
    xn = rng.standard_normal((500, 3))
    tn = _attach(pb, cn, mvn)
    # a theta sequence with repeats: one BUILD per change
    th = res["theta_mcmc"][:, [0, 0, 1, 1, 1, 2, 0, 0, 3, 3]]
    samples = dict(res, theta_mcmc=th)
    n_changes = 1 + int(np.sum(np.any(th[:, 1:] != th[:, :-1], axis=0)))
    a = gm.predict_new(cn, xn, mvn, tn, samples, seed=3, moments=True)
    b = gm.predict_new(cn, xn, mvn, tn, samples, seed=3)
    c = gm.predict_new(cn, xn, mvn, tn, samples, seed=4)
    assert a["n_builds"] == n_changes
    for k in ("w_new", "yhat_new"):
        assert np.array_equal(a[k], b[k]) and not np.array_equal(a[k], c[k])
    for k, kk in (("w_new", "w_new"), ("yhat_new", "yhat_new")):
        assert np.allclose(a[kk + "_mean"], a[k].mean(axis=1), rtol=1e-12, atol=1e-12)
        assert np.allclose(a[kk + "_sd"], a[k].std(axis=1, ddof=1), rtol=1e-10, atol=1e-12)
    # one call over S samples = S calls of one sample each (given the same normals)
    z, eps = rng.standard_normal((500, 10)), rng.standard_normal((500, 10))
    full = gm.predict_new(cn, xn, mvn, tn, samples, moments=True, z=z, eps=eps)
    for s in range(10):
        one = {k: (v[:, s:s + 1] if k in ("theta_mcmc", "tausq_mcmc", "w_mcmc") else v[:, s:s + 1, :]) for k, v in samples.items()
               if k in ("theta_mcmc", "tausq_mcmc", "w_mcmc", "beta_mcmc")}
        o = gm.predict_new(cn, xn, mvn, tn, one, moments=True, z=z[:, s:s + 1], eps=eps[:, s:s + 1])
        assert o["n_builds"] == 1 and o["w_new_sd"].max() == 0.0
        for k in ("w_new", "yhat_new", "mean", "sd"):
            assert np.array_equal(o[k][:, 0], full[k][:, s]), (s, k)
    gm.close()


def test_no_side_effects():
    pb = common.make_problem(1, 625)
    d = pb["d"]
    miss = np.isnan(d["y"])
    tn = _attach(pb, d["coords"][miss], d["mv_id"][miss])
    A, B = common.product_model(pb, keep_H=False), common.product_model(pb, keep_H=False)
    ra, rb = _mcmc(A, pb, seed=3), _mcmc(B, pb, seed=3)
    before = (A.get_loglik_w(0), A.w, A.params())
    B.get_loglik_w(0), B.w, B.params()
    out = A.predict_new(d["coords"][miss], d["X"][miss], d["mv_id"][miss], tn, ra)
    assert out["n_builds"] >= 1
    after = (A.get_loglik_w(0), A.w, A.params())
    assert before[0] == after[0] and np.array_equal(before[1], after[1])
    for k in before[2]:
        assert np.array_equal(before[2][k], after[2][k])
    ra2, rb2 = _mcmc(A, pb, seed=9), _mcmc(B, pb, seed=9)
    for k in ("theta_mcmc", "beta_mcmc", "tausq_mcmc", "w_mcmc", "yhat_mcmc", "paramsd"):
        assert np.array_equal(ra2[k], rb2[k]), k
    assert ra2["n_accepted"] == rb2["n_accepted"]
    A.close()
    B.close()


def test_public_entry_point_and_errors():
    d = synth.make_data(1, 625, missing=0.1, seed=5)
    rng = np.random.default_rng(6)
    cn, xn = rng.random((40, 2)), rng.standard_normal((40, 3))
    kw = dict(mcmc={"keep": 6, "burn": 2, "thin": 1}, seed=3)
    a = sb.spamtree(d["y"], d["X"], d["coords"], **kw)
    b = sb.spamtree(d["y"], d["X"], d["coords"], coords_new=cn, x_new=xn, **kw)
    for k in a:
        if k == "mcmc_time":
            continue
        va, vb = a[k], b[k]
        if isinstance(va, dict):
            assert all(np.array_equal(va[x], vb[x]) for x in va), k
        elif isinstance(va, list):
            assert all(np.array_equal(x, y) for x, y in zip(va, vb)), k
        else:
            assert np.array_equal(np.asarray(va), np.asarray(vb), equal_nan=True), k
    assert b["w_new_mcmc"].shape == (40, 6) and b["yhat_new_mcmc"].shape == (40, 6)
    for k in ("w_new_mean", "w_new_sd", "yhat_new_mean", "yhat_new_sd"):
        assert b[k].shape == (40,) and np.all(np.isfinite(b[k]))

    pb = common.make_problem(1, 625)
    gm = common.product_model(pb, keep_H=False)
    res = _mcmc(gm, pb, keep=3, burn=1, thin=1)
    tn = _attach(pb, cn, None)
    empty = gm.predict_new(np.zeros((0, 2)), None, np.zeros(0, np.int64), {"group": np.zeros(0, np.int64),
                           "parents_ptr": np.zeros(1, np.int64), "parents_idx": np.zeros(0, np.int64)}, res)
    assert empty["w_new"].shape == (0, 3) and empty["n_builds"] == 0
    bad = [dict(tn, group=np.full(40, 10 ** 6)),                                        # group id out of range
           dict(tn, parents_idx=np.full(tn["parents_idx"].size, 10 ** 6)),              # parent id out of range
           dict(tn, parents_idx=tn["parents_idx"][::-1].copy()),                        # not a chain
           dict(tn, parents_ptr=np.zeros_like(tn["parents_ptr"]))]                      # groups without parents
    for t in bad:
        with pytest.raises(sb.SpamTreeError) as ex:
            gm.predict_new(cn, None, None, t, res)
        assert ex.value.code == 1
    with pytest.raises(sb.SpamTreeError) as ex:
        gm.predict_new(cn, None, np.full(40, 5), tn, res)  # mv_id outside 1..q
    assert ex.value.code == 1
    assert np.all(np.isfinite(gm.predict_new(cn, None, None, tn, res)["w_new"]))  # the handle is still usable
    # a theta whose covariance is not positive definite (negative variance): an error, not silent draws
    bad_theta = dict(res, theta_mcmc=np.repeat(np.array([[-1.0], [1.0], [1.0], [6.0]]), 3, axis=1))
    with pytest.raises(sb.SpamTreeError) as ex:
        gm.predict_new(cn, None, None, tn, bad_theta)
    assert ex.value.code == 3
    # the alter slot holds the prediction's BUILD: it is not taken up or read before it is rebuilt
    with pytest.raises(sb.SpamTreeError) as ex:
        gm.accept_make_change()
    assert ex.value.code == 1
    with pytest.raises(sb.SpamTreeError) as ex:
        gm.get_loglik_w(1)
    assert ex.value.code == 1
    gm.get_loglik_comps_w(1)
    gm.get_loglik_w(1)
    gm.accept_make_change()
    with pytest.raises(sb.SpamTreeError) as ex:  # covariates of the new locations are required by spamtree()
        sb.spamtree(d["y"], d["X"], d["coords"], coords_new=cn, **kw)
    assert ex.value.code == 1
    gm.close()

    # a partitioned handle
    t = pb["tree"]
    pl = partition.plan(t, pb["d"]["y"], 2)
    sp = partition.subproblem(pb["d"], t, pl, 0, 2)
    part = dict(sp, allreduce=lambda ptr, count: None)
    pm = sb.SpamTreeMV(sp["y"], sp["X"], sp["coords"], sp["mv_id"], sp["res_is_ref"], None, None, False, sp["block_names"],
                       sp["block_groups"], None, pb["beta"], pb["theta"], pb["tausq"], csr=sp["csr"], partition=part, q=1)
    samples = {"theta_mcmc": pb["theta"][:, None], "beta_mcmc": np.zeros((3, 1, 1)), "tausq_mcmc": np.full((1, 1), .1),
               "w_mcmc": np.zeros((sp["y"].size, 1))}
    with pytest.raises(sb.SpamTreeError) as ex:
        pm.predict_new(cn[:1], None, None, {"group": np.zeros(1, np.int64), "parents_ptr": np.array([0, 1]),
                                            "parents_idx": np.zeros(1, np.int64)}, samples)
    assert ex.value.code == 4
    pm.close()
