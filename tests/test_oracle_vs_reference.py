"""Pins the CPU oracle against the REFERENCE ITSELF: oracle/_ref/libspamtree_ref.so is the reference's own model layer
(spamtree_model.cpp, covariance_functions.cpp, tree_utils.cpp, tree_dep.cpp, mh_adapt.cpp) compiled UNMODIFIED from the
reference package's src/ directory against the Armadillo/Rcpp stand-in of oracle/refshim/ (recipe: `make -C oracle ref`).
The library is built wherever that directory exists (SPAMTREE_REF_SRC, else src/ under BASELINE.json's reference_path);
without it these tests are skipped (the reference's outputs on fixed problems are stored in tests/golden/ref_*.npz and
checked by tests/test_golden_reference.py)."""
import numpy as np
import pytest

import common
from common import orc, relerr
from oracle import ref

pytestmark = pytest.mark.skipif(not ref.available(), reason="oracle/_ref/libspamtree_ref.so not built (the reference sources are not at ref.ref_src())")


def _pair(q, n, missing=.1, limited=False, cell_size=25, proportions=None):
    pb = common.make_problem(q, n, missing=missing, limited=limited, cell_size=cell_size, proportions=proportions)
    d, t = pb["d"], pb["tree"]
    rm = ref.RefModel(d["y"], d["X"], d["coords"], d["mv_id"], t["res_is_ref"], pb["csr"], limited, t["block_names"], t["block_groups"],
                      pb["beta"], pb["theta"], pb["tausq"])
    return pb, rm, common.oracle_model(pb)


@pytest.mark.parametrize("q,n,tol,limited,cell,missing,prop", [
    (1, 625, 2e-9, False, 25, .1, None), (2, 1500, 1e-10, False, 25, .1, None), (3, 3000, 1e-10, False, 25, .1, None),
    (5, 2500, 1e-10, False, 25, .1, None), (3, 900, 1e-10, False, 25, .1, None), (3, 1500, 1e-10, True, 25, .1, None),
    (1, 625, 2e-9, True, 25, .1, None),
    # other cell sizes (rows per reference block), incl. blocks of more than 32 rows
    (2, 1500, 1e-10, False, 9, .1, None), (2, 2000, 1e-10, False, 36, .1, None), (3, 3000, 1e-10, False, 49, .1, None),
    # nothing missing (no prediction blocks), half of the rows missing, strongly imbalanced outcomes (the C4 / C5 proportions)
    (2, 1200, 1e-10, False, 25, 0.0, None), (3, 2400, 1e-10, False, 25, .5, None), (3, 3000, 1e-10, False, 25, .1, (.6, .3, .1)),
    (5, 4000, 1e-10, False, 25, .1, (.55, .25, .10, .07, .03))])
def test_oracle_matches_reference_model_layer(q, n, tol, limited, cell, missing, prop):
    pb, rm, om = _pair(q, n, missing=missing, limited=limited, cell_size=cell, proportions=prop)
    t = pb["tree"]
    nb = t["n_blocks"]
    # integer bookkeeping of the constructor: bit-exact (spamtree_model.cpp:194-420)
    for name in ["blocks_not_empty", "blocks_predicting", "block_is_reference", "block_ct_obs", "n_actual_groups"]:
        assert np.array_equal(rm.geti(name), om.geti(name)), name
    for g in range(int(om.geti("n_actual_groups")[0])):
        assert np.array_equal(rm.geti("u_by_block_groups", g), om.geti("u_by_block_groups", g))
    nchi = np.diff(t["children_ptr"])
    for u in range(nb):
        for name in ["parents_indexing", "children_indexing", "dim_by_parent", "this_is_jth_child"]:
            assert np.array_equal(rm.geti(name, u), om.geti(name, u)), (name, u)
        for c in range(0, nchi[u], max(1, nchi[u] // 4)):
            for which in (0, 1):
                assert np.array_equal(rm.geti("u_is_which_col", u, which, c), om.geti("u_is_which_col", u, which, c))
    rng = np.random.default_rng(7)
    w0 = rng.standard_normal(n) * .5
    rm.w = w0
    om.w = w0
    for slot in (0, 1):   # get_loglik_comps_w_std, spamtree_model.cpp:834-998
        a, b = rm.get_loglik_comps_w(slot), om.get_loglik_comps_w(slot)
        assert a[0] and b[0]
        assert abs(a[1] - b[1]) <= tol * abs(b[1]) and abs(a[2] - b[2]) <= tol * abs(b[2])
    obs, isref = om.geti("block_ct_obs"), om.geti("block_is_reference")
    npar = np.diff(t["parents_ptr"])
    for u in range(nb):
        if obs[u] == 0:
            continue
        if npar[u]:
            assert relerr(rm.get("H", u), om.get("H", u)) <= 10 * tol, ("H", u)
        if isref[u]:
            assert relerr(rm.get("Ri", u), om.get("Ri", u)) <= 10 * tol, ("Ri", u)
            assert relerr(rm.get("prec", u), om.get("prec", u)) <= 10 * tol
            if rm.get("Kxx_inv", u).size:
                assert relerr(rm.get("Kxx_inv", u), om.get("Kxx_inv", u)) <= 100 * tol
        assert relerr(rm.get("ccholprecdiag", u), om.get("ccholprecdiag", u)) <= 10 * tol
    assert relerr(rm.get("logdetCi_comps"), om.get("logdetCi_comps")) <= 10 * tol
    for sweep in range(3):   # gibbs_sample_w_std :1011-1226 (the reference's arma::randn is fed the same z) + get_loglik_w_std :781-826
        z = rng.standard_normal(n)
        rm.deal_with_w(z)
        om.deal_with_w(z)
        assert relerr(rm.w, om.w) <= 100 * tol
        la, lb = rm.get_loglik_w(0), om.get_loglik_w(0)
        assert abs(la[0] - lb[0]) <= 10 * tol * abs(lb[0])
    rm.predict(True)   # predict_std :1234-1358
    om.predict(True)
    assert relerr(rm.w, om.w) <= 100 * tol
    tt = np.linspace(3, 9, q)
    rm.gibbs_sample_tausq(tt)
    om.gibbs_sample_tausq(tt)
    zb = rng.standard_normal((3, q))
    rm.gibbs_sample_beta(zb)   # gibbs_sample_beta :1364-1391, including the row mis-indexing of SURVEY App. D #12
    om.gibbs_sample_beta(zb)
    assert relerr(rm.params()["Bcoeff"], om.params()["Bcoeff"]) <= 100 * tol
    assert relerr(rm.params()["XB"], om.params()["XB"]) <= 100 * tol
    rm.seed(5)
    om.seed(5)
    rm.gibbs_sample_tausq()   # gibbs_sample_tausq :1393-1417 with R::rgamma fed from the shared host stream
    om.gibbs_sample_tausq()
    assert relerr(rm.params()["tausq_inv"], om.params()["tausq_inv"]) <= 100 * tol
    # accept_make_change :1432-1435
    th2 = pb["theta"] * (1 + .01 * rng.standard_normal(pb["theta"].size))
    for m in (rm, om):
        m.theta_update(1, th2)
    a, b = rm.get_loglik_comps_w(1), om.get_loglik_comps_w(1)
    assert a[0] == b[0] and abs(a[1] - b[1]) <= 10 * tol * abs(b[1])
    for m in (rm, om):
        m.accept_make_change()
    z = rng.standard_normal(n)
    rm.deal_with_w(z)
    om.deal_with_w(z)
    assert relerr(rm.w, om.w) <= 100 * tol
    rm.close()
    om.close()


def test_reference_standalone_exports():
    assert list(ref.kthresholds(np.arange(1, 101.0), 4)) == [26, 51, 76]
    rng = np.random.default_rng(0)
    x = rng.random(1234)
    assert np.array_equal(ref.kthresholds(x, 17), orc.kthresholds(x, 17))
    om_ = rng.integers(0, 50, size=(60, 5))
    fv, tv = np.arange(1, 41), rng.integers(0, 30, size=40)
    assert np.array_equal(ref.number_revalue(om_, fv, tv), orc.number_revalue(om_, fv, tv))
    c1, c2 = rng.random((57, 2)), rng.random((31, 2))
    m1, m2 = rng.integers(1, 4, 57), rng.integers(1, 4, 31)
    D = np.array([[0, 1, 2], [1, 0, 1.5], [2, 1.5, 0.0]])
    a3 = ([1, 1.5, .8], [.1, .51, .3], [1, 2, 3], [2, .5, 5.0], D)
    assert relerr(ref.cross_covariance_ag10(c1, m1, c2, m2, *a3), orc.cross_covariance_ag10(c1, m1, c2, m2, *a3)) <= 1e-14


def test_reference_cholesky_failure_is_a_rejection():
    pb, rm, om = _pair(3, 900)
    assert rm.get_loglik_comps_w(0)[0]
    bad = pb["theta"].copy()
    bad[12:] = [1e-3, 1e-3, 999.0]
    bad[0:3] = [30, -30, 30]
    for m in (rm, om):
        m.theta_update(1, bad)
    assert rm.get_loglik_comps_w(1)[0] == om.get_loglik_comps_w(1)[0]
    rm.close()
    om.close()
