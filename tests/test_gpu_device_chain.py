"""The device-resident chain (rng_mode 1: proposal, accept decision, slot swap, RAM adaptation, tausq / beta draws, yhat and
the saves all on the device, no host round trip per iteration) against a HOST REPLAY: the same run driven call by call
through the reference-named operations of the C ABI (which are pinned to the oracle and to the reference's own driver),
fed the random numbers the device drew (tests/philox_host.py restates the device streams)."""
import numpy as np
import pytest

import common
import philox_host as ph
from common import relerr
import spamtree_b200 as sb
from spamtree_b200 import synth

pytestmark = pytest.mark.gpu


def _replay(pb, bounds, sd0, keep, burn, thin, seed, faithful, adapting=True, predicts=True):
    """spamtree_fit.cpp:167-391 on the host-driven path with the device's random numbers"""
    d = pb["d"]
    y, mv, q, n = d["y"], d["mv_id"], pb["q"], pb["n"]
    gm = common.product_model(pb, keep_H=False)
    gm.get_loglik_comps_w(0)
    gm.get_loglik_comps_w(1)
    obs = np.isfinite(y)
    p = d["X"].shape[1]
    npar = pb["theta"].size
    param = pb["theta"].copy()
    predict_param = param.copy()
    psd = np.linalg.cholesky(sd0)
    Us, alphas = [], []
    out = {"theta": [], "beta": [], "tausq": [], "w": [], "yhat": [], "acc": 0}
    rows = np.arange(n, dtype=np.uint64)
    for m in range(thin * keep + burn):
        saved = m - burn >= 0 and (m - burn) % thin == 0
        gm.deal_with_w(ph.normal(seed, rows, m))
        ll_cur = gm.get_loglik_w(0)[0]
        U = ph.normal(seed, ph.K_STREAM_U + np.arange(npar, dtype=np.uint64), m)
        new_param, jac, _ = sb.mh_propose(param, bounds, psd, U)
        gm.theta_update(1, new_param)
        ok, ll_new, _ = gm.get_loglik_comps_w(1)
        logaccept = ll_new - ll_cur + jac
        u = float(ph.uniform(seed, ph.K_STREAM_ACCEPT, m)[0])
        if sb.do_I_accept(logaccept, u) and ok:
            gm.accept_make_change()
            param = new_param
            out["acc"] += 1
        if adapting:
            Us.append(U)
            alphas.append((1.0 if ok else 0.0) * np.exp(logaccept))
            psd, _ = sb.ram_adapt(sd0, np.array(Us), np.array(alphas))
        need = bool(np.any(np.abs(param - predict_param) > 1e-5))
        if saved and predicts:
            gm.predict(need)
            predict_param = param.copy()
        pr = gm.params()
        w = gm.w
        tq = np.zeros(q)
        for j in range(q):
            sel = obs & (mv == j + 1)
            bcore = float(np.sum((y[sel] - pr["XB"][sel] - w[sel]) ** 2))
            tq[j] = ph.gamma(seed, ph.K_STREAM_GAMMA + (j << 32), m, 2.01 + sel.sum() / 2.0, 1.0 / (1.0 + .5 * bcore))
        gm.gibbs_sample_tausq(tq)
        zb = np.array([[float(ph.normal(seed, ph.K_STREAM_BETA + (j << 32) + a, m)[0]) for j in range(q)] for a in range(p)])
        gm.gibbs_sample_beta(zb, faithful)
        if saved:
            pr = gm.params()
            out["theta"].append(param.copy())
            out["beta"].append(pr["Bcoeff"].copy())
            out["tausq"].append(1.0 / pr["tausq_inv"])
            out["w"].append(gm.w)
            e = ph.normal(seed, rows, ph.K_COUNTER_YHAT + m + 1)
            out["yhat"].append(pr["XB"] + out["w"][-1] + e / np.sqrt(pr["tausq_inv"][mv - 1]))
    out["paramsd"] = psd
    gm.close()
    return out


# early: ST_EARLY_LEVELS, the number of tree levels whose BUILD runs on the second stream underneath the Gibbs sweep (None: the
# library's choice; 0: sequential; 99: every level, the childless level's log-density pieces then come from its parked Z)
@pytest.mark.parametrize("q,n,sd,keep,burn,thin,faithful,early", [(1, 625, 1e-2, 12, 45, 2, True, None), (2, 1200, 1e-7, 30, 30, 1, False, None),
                                                                  (3, 1500, 1e-7, 16, 0, 2, True, None), (3, 1500, 1e-7, 16, 0, 2, True, "0"),
                                                                  (3, 1500, 1e-7, 16, 0, 2, True, "99"), (1, 625, 1e-2, 12, 45, 2, True, "99"),
                                                                  (2, 6000, 1e-7, 10, 10, 1, False, "99")])
def test_device_chain_equals_host_replay(q, n, sd, keep, burn, thin, faithful, early, monkeypatch):
    if early is not None:
        monkeypatch.setenv("ST_EARLY_LEVELS", early)
    pb = common.make_problem(q, n)
    bounds = synth.default_bounds(q)
    npar = pb["theta"].size
    sd0 = np.eye(npar) * sd
    seed = 77 + q
    gm = common.product_model(pb, keep_H=False)
    r = gm.mcmc(bounds, sd0, keep, burn, thin, adapting=True, faithful_beta_index=faithful, rng_mode=1, seed=seed)
    gm.close()
    h = _replay(pb, bounds, sd0, keep, burn, thin, seed, faithful)
    total = thin * keep + burn
    assert r["n_accepted"] == h["acc"] and 0 < h["acc"] < total
    th, be = np.array(h["theta"]).T, np.array(h["beta"]).transpose(1, 0, 2)
    err = {"theta": relerr(r["theta_mcmc"], th), "beta": relerr(r["beta_mcmc"], be), "tausq": relerr(r["tausq_mcmc"], np.array(h["tausq"]).T),
           "paramsd": relerr(r["paramsd"], h["paramsd"]), "w": relerr(r["w_mcmc"], np.array(h["w"]).T),
           "yhat": relerr(r["yhat_mcmc"], np.array(h["yhat"]).T)}
    print(f"device-resident chain vs host replay (q={q}, {total} iterations, {h['acc']} accepted):", {k: f"{v:.2e}" for k, v in err.items()})
    # same kernels on both sides; only the scalar glue runs in different places (device vs host libm): agreement far below
    # the 1e-9 contract even after the chain's amplification
    assert all(v <= 1e-9 for v in err.values()), err


@pytest.mark.parametrize("ncol", [1, 2])
def test_device_chain_with_one_or_two_regressors(ncol):
    """p < 3 with q > 1: every outcome's work arrays of the beta step must stay its own (the layout once assumed p >= 3)"""
    pb = common.make_problem(2, 1200)
    pb["d"] = dict(pb["d"], X=np.ascontiguousarray(pb["d"]["X"][:, :ncol]))
    pb["beta"] = np.zeros(ncol)
    bounds, npar = synth.default_bounds(2), pb["theta"].size
    sd0 = np.eye(npar) * 1e-7
    gm = common.product_model(pb, keep_H=False)
    r = gm.mcmc(bounds, sd0, 12, 6, 1, adapting=True, faithful_beta_index=False, rng_mode=1, seed=21)
    gm.close()
    h = _replay(pb, bounds, sd0, 12, 6, 1, 21, False)
    assert r["n_accepted"] == h["acc"]
    err = {"beta": relerr(r["beta_mcmc"], np.array(h["beta"]).transpose(1, 0, 2)), "tausq": relerr(r["tausq_mcmc"], np.array(h["tausq"]).T),
           "w": relerr(r["w_mcmc"], np.array(h["w"]).T), "yhat": relerr(r["yhat_mcmc"], np.array(h["yhat"]).T)}
    assert all(v <= 1e-9 for v in err.values()), err


@pytest.mark.parametrize("keep,burn,thin", [(1, 0, 1), (2, 0, 1), (1, 2, 1), (2, 1, 3)])
def test_very_short_device_chains(keep, burn, thin):
    """one, two, three ... iterations: the first iteration draws its own proposal and normals, every other one finds them drawn
    by its predecessor, the last one draws none — the alter slot must still hold the proposal that was built"""
    pb = common.make_problem(1, 625)
    bounds, npar = synth.default_bounds(1), pb["theta"].size
    sd0 = np.eye(npar) * 1e-2
    gm = common.product_model(pb, keep_H=False)
    r = gm.mcmc(bounds, sd0, keep, burn, thin, adapting=True, faithful_beta_index=True, rng_mode=1, seed=9)
    # after the run the host-driven operations continue from the chain's state: the alter slot is the last proposal's BUILD
    ll_alt = gm.get_loglik_comps_w(1)
    gm.close()
    h = _replay(pb, bounds, sd0, keep, burn, thin, 9, True)
    assert r["n_accepted"] == h["acc"]
    err = {"theta": relerr(r["theta_mcmc"], np.array(h["theta"]).T), "beta": relerr(r["beta_mcmc"], np.array(h["beta"]).transpose(1, 0, 2)),
           "w": relerr(r["w_mcmc"], np.array(h["w"]).T), "yhat": relerr(r["yhat_mcmc"], np.array(h["yhat"]).T)}
    assert all(v <= 1e-9 for v in err.values()), err
    assert ll_alt[0] and np.isfinite(ll_alt[1])


def test_device_chain_is_reproducible_and_seed_dependent():
    pb = common.make_problem(2, 900)
    bounds, npar = synth.default_bounds(2), pb["theta"].size
    runs = []
    for seed in (5, 5, 6):
        gm = common.product_model(pb, keep_H=False)
        runs.append(gm.mcmc(bounds, np.eye(npar) * 1e-7, 10, 10, 1, rng_mode=1, seed=seed, save_yhat=False))
        gm.close()
    assert np.array_equal(runs[0]["theta_mcmc"], runs[1]["theta_mcmc"]) and np.array_equal(runs[0]["w_mcmc"], runs[1]["w_mcmc"])
    assert not np.array_equal(runs[0]["w_mcmc"], runs[2]["w_mcmc"])


def test_device_chain_without_graph_matches_graph(monkeypatch, tmp_path):
    """ST_GRAPH=0 enqueues every iteration kernel by kernel; the CUDA-graph replay must give bit-identical chains"""
    import os, subprocess, sys
    code = ("import sys; sys.path.insert(0, 'tests'); import numpy as np, common; from spamtree_b200 import synth;"
            "pb = common.make_problem(2, 900); gm = common.product_model(pb, keep_H=False);"
            "r = gm.mcmc(synth.default_bounds(2), np.eye(pb['theta'].size) * 1e-7, 12, 8, 1, rng_mode=1, seed=3, save_yhat=False);"
            "np.save(sys.argv[1], np.concatenate([r['theta_mcmc'].ravel(), r['w_mcmc'].ravel(), r['beta_mcmc'].ravel()]))")
    outs = []
    for g in ("1", "0"):
        path = str(tmp_path / f"graph_{g}.npy")
        env = dict(os.environ, ST_GRAPH=g)
        subprocess.run([sys.executable, "-c", code, path], check=True, env=env, cwd=common.ROOT)
        outs.append(np.load(path))
    assert np.array_equal(outs[0], outs[1])
