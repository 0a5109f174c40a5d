"""Parity of the CUDA hot path (through the C ABI) against the CPU oracle on identical seeded inputs.
Contract (BASELINE.json north_star / SURVEY §8c): H, Ri, log-density at fixed theta, Gibbs conditional mean and
covariance <= 1e-9 relative (max-norm per block); w identical to <= 1e-9 given the same z."""
import numpy as np
import pytest

import common
from common import orc, relerr
from dense_twin import Twin

pytestmark = pytest.mark.gpu
TOL = 1e-9

CASES = [(1, 625, .1), (1, 2500, .1), (2, 2000, .1), (3, 3000, .1), (5, 4000, .15), (3, 1200, 0.0), (1, 30, .1), (2, 9, 0.0),
         (3, 3000, .1, True), (1, 625, .1, True),   # 4th entry: limited_tree = TRUE (make_edges_limited, spamtree_model.cpp:901-903)
         # 5th entry: cell_size of spamtree() (R/spamtree_fit.R:229-233) = rows per reference block: blocks smaller than the
         # default 25, and blocks of more than 32 rows, which take the kernels' general (not register-resident) Cholesky paths
         (2, 1500, .1, False, 9), (1, 1200, .1, False, 16), (2, 2500, .1, False, 36), (3, 4000, .1, False, 49),
         # half of the rows missing; 6th entry: strongly imbalanced outcome proportions (those of C4 / C5)
         (3, 2400, .5), (3, 3000, .1, False, 25, (.6, .3, .1)), (5, 4000, .1, False, 25, (.55, .25, .10, .07, .03))]


def _case_id(c):
    return (f"q{c[0]}_n{c[1]}_miss{c[2]}" + ("_limited" if len(c) > 3 and c[3] else "") + (f"_cell{c[4]}" if len(c) > 4 and c[4] != 25 else "") +
            ("_imbalanced" if len(c) > 5 else ""))


@pytest.fixture(scope="module", params=CASES, ids=_case_id)
def pair(request):
    q, n, missing = request.param[:3]
    pb = common.make_problem(q, n, missing=missing, limited=len(request.param) > 3 and request.param[3],
                             cell_size=request.param[4] if len(request.param) > 4 else 25,
                             proportions=request.param[5] if len(request.param) > 5 else None)
    gm, om = common.product_model(pb), common.oracle_model(pb)
    w0 = np.random.default_rng(7).standard_normal(n) * .5
    gm.w = w0
    om.w = w0
    yield pb, gm, om
    gm.close()
    om.close()


def test_build_H_Ri_logdensity(pair):
    pb, gm, om = pair
    nb = pb["tree"]["n_blocks"]
    for slot in (0, 1):
        okg, llg, ldg = gm.get_loglik_comps_w(slot)
        oko, llo, ldo = om.get_loglik_comps_w(slot)
        assert okg and oko
        assert abs(llg - llo) <= TOL * abs(llo) and abs(ldg - ldo) <= TOL * abs(ldo)
    obs, isref = om.geti("block_ct_obs"), om.geti("block_is_reference")
    npar = np.diff(pb["tree"]["parents_ptr"])
    for u in range(nb):
        if obs[u] == 0:
            continue
        if npar[u]:
            assert relerr(gm.node_state("H", u), om.get("H", u)) <= TOL, ("H", u)
        ref = om.get("Ri", u) if isref[u] else om.get("ccholprecdiag", u)
        assert relerr(gm.node_state("Ri", u), ref) <= TOL, ("Ri", u)
    assert relerr(gm.node_state("logdetCi_comps"), om.get("logdetCi_comps")) <= TOL
    assert relerr(gm.node_state("loglik_w_comps"), om.get("loglik_w_comps")) <= TOL


def test_gibbs_conditionals_and_draw(pair):
    pb, gm, om = pair
    n, nb = pb["n"], pb["tree"]["n_blocks"]
    gm.get_loglik_comps_w(0)
    om.get_loglik_comps_w(0)
    obs, isref = om.geti("block_ct_obs"), om.geti("block_is_reference")
    rng = np.random.default_rng(8)
    worst_cond = 1.0
    for sweep in range(3):
        # the third sweep draws no noise: w is then the conditional MEAN of every block as the sampler realises it
        # (Sc'(Sc Smu_tot), spamtree_model.cpp:1086) — compared directly, no inverse formed by the test
        z = rng.standard_normal(n) if sweep < 2 else np.zeros(n)
        gm.deal_with_w(z)
        om.deal_with_w(z)
        assert relerr(gm.w, om.w) <= TOL
        for u in range(nb):
            if obs[u] == 0:
                continue
            Sg, So = gm.node_state("Sigi_tot", u), om.get("Sigi_tot", u)
            Mg, Mo = gm.node_state("Smu_tot", u), om.get("Smu_tot", u)
            assert relerr(Sg, So) <= TOL and relerr(Mg, Mo) <= TOL
            if isref[u]:  # conditional covariance Sigi_tot^-1 and mean Sigi_tot^-1 Smu_tot, inverted HERE by numpy: the
                # inversion amplifies the (<= 1e-9) difference of the two precisions by the condition number of Sigi_tot
                m = Mo.size
                So2 = So.reshape(m, m)
                cond = float(np.linalg.cond(So2))
                worst_cond = max(worst_cond, cond)
                Cg, Co = np.linalg.inv(Sg.reshape(m, m)), np.linalg.inv(So2)
                bound = max(TOL, 4 * cond * max(relerr(Sg, So), relerr(Mg, Mo), 1e-16))
                assert relerr(Cg, Co) <= bound and relerr(Cg @ Mg, Co @ Mo) <= bound, (u, cond)
                assert relerr(Cg, Co) <= 100 * TOL and relerr(Cg @ Mg, Co @ Mo) <= 100 * TOL
            else:
                assert relerr(Mg / Sg, Mo / So) <= TOL
        lg, lo = gm.get_loglik_w(0), om.get_loglik_w(0)
        assert abs(lg[0] - lo[0]) <= TOL * abs(lo[0]) and abs(lg[1] - lo[1]) <= TOL * abs(lo[1])
    print(f"largest condition number of a block's conditional precision: {worst_cond:.2e}")


def test_predict_beta_tausq(pair):
    pb, gm, om = pair
    q = pb["q"]
    rng = np.random.default_rng(9)
    z = rng.standard_normal(pb["n"])
    gm.deal_with_w(z)
    om.deal_with_w(z)
    gm.predict(True)
    om.predict(True)
    assert relerr(gm.w, om.w) <= TOL
    gm.predict(False)   # H of the prediction blocks is reused (spamtree_model.cpp:1256)
    om.predict(False)
    assert relerr(gm.w, om.w) <= TOL
    t = np.linspace(3, 9, q)
    gm.gibbs_sample_tausq(t)
    om.gibbs_sample_tausq(t)
    zb = rng.standard_normal((3, q))
    gm.gibbs_sample_beta(zb, True)   # reference indexing quirk (SURVEY App. D #12)
    om.gibbs_sample_beta(zb)
    pg, po = gm.params(), om.params()
    assert relerr(pg["Bcoeff"], po["Bcoeff"]) <= TOL and relerr(pg["XB"], po["XB"]) <= TOL
    gm.seed(5)
    om.seed(5)
    gm.gibbs_sample_tausq()
    om.gibbs_sample_tausq()
    assert relerr(gm.params()["tausq_inv"], om.params()["tausq_inv"]) <= TOL
    # corrected beta indexing against an oracle built with that flag
    om2 = common.oracle_model(pb, flags=orc.FLAG_PROBES | orc.FLAG_CORRECT_BETA_INDEX)
    om2.w = gm.w
    om2.set_tausq_inv(gm.params()["tausq_inv"])
    gm.gibbs_sample_beta(zb, False)
    om2.gibbs_sample_beta(zb)
    assert relerr(gm.params()["Bcoeff"], om2.params()["Bcoeff"]) <= TOL
    om2.close()
    gm.gibbs_sample_beta(zb, True)   # leave the pair in the same state for the tests that follow
    om.gibbs_sample_beta(zb)
    assert relerr(gm.params()["XB"], om.params()["XB"]) <= TOL


def test_swap_and_two_slots(pair):
    pb, gm, om = pair
    th2 = pb["theta"] * (1 + .01 * np.random.default_rng(3).standard_normal(pb["theta"].size))
    for m in (gm, om):
        m.theta_update(1, th2)
    rg, ro = gm.get_loglik_comps_w(1), om.get_loglik_comps_w(1)
    assert rg[0] and ro[0] and abs(rg[1] - ro[1]) <= TOL * abs(ro[1])
    for m in (gm, om):
        m.accept_make_change()
    lg, lo = gm.get_loglik_w(0), om.get_loglik_w(0)   # param_data is now the theta-2 state
    assert abs(lg[0] - rg[1]) <= 1e-12 * abs(rg[1])
    assert abs(lg[0] - lo[0]) <= TOL * abs(lo[0])
    z = np.random.default_rng(4).standard_normal(pb["n"])
    gm.deal_with_w(z)
    om.deal_with_w(z)
    assert relerr(gm.w, om.w) <= TOL
    for m in (gm, om):
        m.accept_make_change()


def test_lockstep_chain_matches_oracle_chain():
    """spamtree_mv_mcmc (spamtree_fit.cpp:167-391) run on both sides with the same host random stream"""
    from spamtree_b200 import synth
    for q, n in [(1, 625), (2, 1500)]:
        pb = common.make_problem(q, n)
        gm, om = common.product_model(pb), common.oracle_model(pb)
        npar = pb["theta"].size
        bounds = synth.default_bounds(q)
        kw = dict(keep=15, burn=70, thin=2, adapting=True, seed=21)
        sd = np.eye(npar) * (.01 if q == 1 else 2e-4)
        rg = gm.mcmc(bounds, sd, rng_mode=0, **kw)
        ro = om.mcmc(bounds, sd, **kw)
        assert rg["n_accepted"] == ro["n_accepted"] and rg["n_accepted"] >= 1
        for k in ("theta_mcmc", "beta_mcmc", "tausq_mcmc", "w_mcmc", "yhat_mcmc", "paramsd"):
            assert relerr(rg[k], ro[k]) <= TOL, (k, relerr(rg[k], ro[k]))
        gm.close()
        om.close()


@pytest.mark.parametrize("ncol", [1, 2])
def test_lockstep_chain_with_one_or_two_regressors(ncol):
    """p = 1 (intercept-only design) and p = 2 with q = 2 against the oracle, which tests/test_reference_driver.py pins to the
    reference's own driver at these sizes"""
    from spamtree_b200 import synth
    pb = common.make_problem(2, 900)
    pb["d"] = dict(pb["d"], X=np.ascontiguousarray(pb["d"]["X"][:, :ncol]))
    pb["beta"] = np.zeros(ncol)
    gm, om = common.product_model(pb), common.oracle_model(pb)
    bounds, npar = synth.default_bounds(2), pb["theta"].size
    kw = dict(keep=20, burn=0, thin=1, adapting=True, seed=4)
    rg = gm.mcmc(bounds, np.eye(npar) * 1e-7, rng_mode=0, **kw)
    ro = om.mcmc(bounds, np.eye(npar) * 1e-7, **kw)
    assert rg["n_accepted"] == ro["n_accepted"] and rg["beta_mcmc"].shape[0] == ncol
    for k in ("theta_mcmc", "beta_mcmc", "tausq_mcmc", "w_mcmc", "yhat_mcmc"):
        assert relerr(rg[k], ro[k]) <= TOL, (k, relerr(rg[k], ro[k]))
    gm.close()
    om.close()


def _batch_means_se(x, nb=20):
    x = np.asarray(x, dtype=np.float64)
    L = x.size // nb
    return float(x[:L * nb].reshape(nb, L).mean(axis=1).std(ddof=1) / np.sqrt(nb))


def test_posterior_summaries_are_statistically_equivalent_with_device_rng():
    """north_star: 'posterior summaries must be statistically equivalent at a fixed seed'.  With rng_mode = 1 the product
    draws the n-long normal vectors on the device (Philox), so its chain cannot be compared with the oracle's draw by draw
    (test_lockstep_chain_matches_oracle_chain does that for rng_mode = 0): the two chains are two MCMC estimates of the same
    posterior and must agree within Monte-Carlo error (batch-means standard errors).  C1 shape (README example: q = 1,
    n = 625, 10 % missing), 500 burn-in + 1500 kept iterations, RAM adaptation on.  Thresholds calibrated on two oracle
    chains with different seeds (z <= 1.8 there); theta[1], theta[2] do not enter the q = 1 covariance (cexpcov,
    covariance_functions.cpp:95-111 uses ai1[0] and thetamv[0] only) and wander over their prior: not compared."""
    from spamtree_b200 import synth
    pb = common.make_problem(1, 625)
    gm, om = common.product_model(pb), common.oracle_model(pb)
    npar = pb["theta"].size
    bounds, sd = synth.default_bounds(1), np.eye(npar) * .01
    kw = dict(keep=1500, burn=500, thin=1, adapting=True, sample_predicts=False)
    rg = gm.mcmc(bounds, sd, rng_mode=1, seed=11, save_w=True, save_yhat=False, **kw)
    ro = om.mcmc(bounds, sd, seed=12, **kw)
    gm.close()
    om.close()
    assert rg["n_accepted"] > 150 and ro["n_accepted"] > 150  # both chains move (RAM adaptation targets 23 %)
    assert abs(rg["n_accepted"] - ro["n_accepted"]) < 0.35 * ro["n_accepted"]
    pairs = [(f"beta[{a}]", rg["beta_mcmc"][a, :, 0], ro["beta_mcmc"][a, :, 0]) for a in range(3)]
    pairs += [("tausq", rg["tausq_mcmc"][0], ro["tausq_mcmc"][0]), ("sigmasq = theta[0]", rg["theta_mcmc"][0], ro["theta_mcmc"][0]),
              ("phi = theta[3]", rg["theta_mcmc"][3], ro["theta_mcmc"][3])]
    for name, a, b in pairs:
        se = np.hypot(_batch_means_se(a), _batch_means_se(b))
        assert abs(a.mean() - b.mean()) <= 4.5 * se, (name, a.mean(), b.mean(), se)
        if name.startswith(("beta", "tausq")):  # same posterior spread (the Gibbs-sampled, well-mixing parameters)
            assert 0.5 <= (a.std() + 1e-300) / (b.std() + 1e-300) <= 2.0, (name, a.std(), b.std())
    mg, mo = rg["w_mcmc"].mean(axis=1), ro["w_mcmc"].mean(axis=1)  # posterior mean of the latent field, all 625 rows
    assert np.corrcoef(mg, mo)[0, 1] >= 0.995
    assert np.sqrt(np.mean((mg - mo) ** 2)) <= 0.1 * mo.std()


def test_deferred_backward_half_of_childless_levels():
    """with keep_H = 0 the childless non-reference level gets only the forward half of BUILD (log-density); G appears when
    the slot is taken up.  Everything downstream must equal the eager model (keep_H = 1 never defers)."""
    pb = common.make_problem(3, 6000)
    ge, gd = common.product_model(pb, keep_H=True), common.product_model(pb, keep_H=False)
    rng = np.random.default_rng(4)
    n = pb["d"]["y"].size
    w0 = rng.standard_normal(n) * .3
    th2 = pb["theta"] * (1 + .01 * rng.standard_normal(pb["theta"].size))
    for g in (ge, gd):
        g.w = w0
        g.get_loglik_comps_w(0)
        g.theta_update(1, th2)
    a, b = ge.get_loglik_comps_w(1), gd.get_loglik_comps_w(1)
    assert a[0] and b[0] and abs(a[1] - b[1]) <= 1e-11 * abs(a[1]) and abs(a[2] - b[2]) <= 1e-12 * abs(a[2])
    for g in (ge, gd):
        g.accept_make_change()
    t = pb["tree"]
    nchi, npar = np.diff(t["children_ptr"]), np.diff(t["parents_ptr"])
    obs = ge.index("block_ct_obs")
    leaves = [u for u in range(t["n_blocks"]) if nchi[u] == 0 and npar[u] > 0 and obs[u] > 0][:40]
    assert leaves
    for u in leaves:
        assert np.array_equal(ge.node_state("G", u), gd.node_state("G", u)), u
        assert np.array_equal(ge.node_state("Ri", u), gd.node_state("Ri", u)), u
    z = rng.standard_normal(n)
    for g in (ge, gd):
        g.deal_with_w(z)
    assert np.array_equal(ge.w, gd.w)
    la, lb = ge.get_loglik_w(0), gd.get_loglik_w(0)
    assert abs(la[0] - lb[0]) <= 1e-12 * abs(la[0])
    # a rejected proposal leaves the current slot untouched
    for g in (ge, gd):
        g.theta_update(1, pb["theta"])
        g.get_loglik_comps_w(1)
        g.deal_with_w(z)
    assert np.array_equal(ge.w, gd.w)
    ge.close()
    gd.close()


def test_asynchronous_save_of_w_equals_the_synchronous_one():
    """saved iterations without yhat copy w to the caller's buffer on a second stream while the next iteration runs
    (st_model.cu: Model::save_rows, CopyOut); the saved draws must be the very same numbers as with the synchronous path"""
    from spamtree_b200 import synth
    pb = common.make_problem(3, 4000)
    npar = pb["theta"].size
    bounds, sd = synth.default_bounds(3), np.eye(npar) * 1e-4
    res = []
    for yhat in (True, False):
        gm = common.product_model(pb)
        res.append(gm.mcmc(bounds, sd, keep=6, burn=3, thin=2, adapting=True, seed=9, rng_mode=0, save_w=True, save_yhat=yhat))  # mode 0: the host stream is consumed identically with and without yhat
        gm.close()
    assert res[0]["w_mcmc"].shape == res[1]["w_mcmc"].shape and np.abs(res[0]["w_mcmc"]).max() > 0
    assert np.array_equal(res[0]["w_mcmc"], res[1]["w_mcmc"])
    assert np.array_equal(res[0]["theta_mcmc"], res[1]["theta_mcmc"])


def test_cholesky_failure_rejects_without_error():
    """BUILD returns ok = 0 (spamtree_model.cpp:971-982) and the slot recovers; never an exception"""
    pb = common.make_problem(3, 900)
    gm, om = common.product_model(pb), common.oracle_model(pb)
    assert gm.get_loglik_comps_w(0)[0]
    ll_before = gm.get_loglik_comps_w(1)[1]
    bad = pb["theta"].copy()
    bad[12:] = [1e-3, 1e-3, 999.0]
    bad[0:3] = [30, -30, 30]
    for m in (gm, om):
        m.theta_update(1, bad)
    okg, llg, _ = gm.get_loglik_comps_w(1)
    oko = om.get_loglik_comps_w(1)[0]
    assert okg == oko
    if not okg:
        assert llg == ll_before  # loglik_w of the slot is left untouched on failure
    gm.theta_update(1, pb["theta"])
    assert gm.get_loglik_comps_w(1)[0]
    z = np.random.default_rng(1).standard_normal(pb["n"])
    gm.deal_with_w(z)   # the param slot was never touched
    gm.close()
    om.close()


def test_cross_covariance_ag10_on_gpu():
    import spamtree_b200 as sb
    xl = np.linspace(0, 1, 10)
    g = np.array([(a, b) for b in xl for a in xl])
    coords = np.vstack([g, g])
    mv = np.r_[np.ones(100, int), 2 * np.ones(100, int)]
    args = ([1, 1.5], [.1, .51], [1, 2], [5.0], np.array([[0, 1.0], [1.0, 0]]))
    CC = sb.CrossCovarianceAG10(coords, mv, coords, mv, *args)
    assert np.allclose(np.diag(CC)[:100], 1.01, rtol=0, atol=1e-14) and np.allclose(np.diag(CC)[100:], 2.5101, rtol=0, atol=1e-14)
    assert relerr(CC, orc.cross_covariance_ag10(coords, mv, coords, mv, *args)) <= 1e-13
    rng = np.random.default_rng(0)
    c1, c2 = rng.random((57, 2)), rng.random((31, 2))
    m1, m2 = rng.integers(1, 4, 57), rng.integers(1, 4, 31)
    D = np.array([[0, 1, 2], [1, 0, 1.5], [2, 1.5, 0.0]])
    a3 = ([1, 1.5, .8], [.1, .51, .3], [1, 2, 3], [2, .5, 5.0], D)
    assert relerr(sb.CrossCovarianceAG10(c1, m1, c2, m2, *a3), orc.cross_covariance_ag10(c1, m1, c2, m2, *a3)) <= 1e-13
    with pytest.raises(sb.SpamTreeError):
        sb.CrossCovarianceAG10(c1, np.ones(57, int), c2, np.ones(31, int), [1], [1], [1], [1], np.zeros((1, 1)))


def test_gpu_matches_dense_math_directly():
    """independent of the oracle: H, Ri, log-density against scipy-free dense numpy on a small tree (the dense float64
    solve of numpy is itself only good to ~cond * eps, hence one digit of slack on H and Ri; the full-size tests compare
    the deepest blocks with extended-precision dense algebra at 1e-9)"""
    pb = common.make_problem(3, 900)
    gm, tw = common.product_model(pb), Twin(pb)
    w = np.random.default_rng(2).standard_normal(900)
    gm.w = w
    ok, ll, _ = gm.get_loglik_comps_w(0)
    assert ok and abs(ll - tw.loglik(w)) <= TOL * abs(ll)
    for u in range(tw.nb):
        if tw.obs[u] == 0:
            continue
        H, Ri = tw.block(u)
        m = tw.rows[u].size
        if H.shape[1]:
            assert relerr(gm.node_state("H", u).reshape(-1, m).T, H) <= 10 * TOL
        got = gm.node_state("Ri", u)
        assert relerr(got.reshape(m, m).T if tw.isref[u] else got, Ri) <= 10 * TOL
    gm.close()


def test_unsupported_inputs_fail_loudly():
    import spamtree_b200 as sb
    pb = common.make_problem(1, 625)
    d, t = pb["d"], pb["tree"]
    with pytest.raises(sb.SpamTreeError) as e:
        sb.SpamTreeMV(d["y"], d["X"], d["coords"], d["mv_id"], t["res_is_ref"], None, None, True, t["block_names"],
                      t["block_groups"], None, pb["beta"], pb["theta"], pb["tausq"], csr=pb["csr"])
    assert e.value.code == 4
    bad = list(pb["csr"])
    bad[3] = bad[3].copy()
    bad[3][-1] = 0  # break a parent chain
    with pytest.raises(sb.SpamTreeError):
        sb.SpamTreeMV(d["y"], d["X"], d["coords"], d["mv_id"], t["res_is_ref"], None, None, False, t["block_names"],
                      t["block_groups"], None, pb["beta"], pb["theta"], pb["tausq"], csr=tuple(bad))
