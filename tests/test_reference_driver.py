"""Pins the DAG builders, the Metropolis-Hastings glue and the whole MCMC driver to the REFERENCE'S OWN CODE:
oracle/_ref/libspamtree_ref.so now also holds spamtree_fit.cpp (the driver spamtree_mv_mcmc itself) and tree_dep.cpp's
make_edges / make_edges_limited / part_axis_parallel_lmt with their return values retained by the Rcpp::List stand-in
(oracle/refshim/RcppArmadillo.h).  Product (host code behind the C ABI — no GPU needed) and oracle are both compared with it."""
import numpy as np
import pytest

import common
from common import orc, relerr
from oracle import ref
import spamtree_b200 as sb
from spamtree_b200 import synth

pytestmark = pytest.mark.skipif(not ref.available(), reason="oracle/_ref/libspamtree_ref.so not built (the reference sources are not at ref.ref_src())")


def _same_lists(a, b):
    return len(a) == len(b) and all(np.array_equal(np.asarray(x, dtype=np.int64), np.asarray(y, dtype=np.int64)) for x, y in zip(a, b))


@pytest.mark.parametrize("q,n,missing,cell", [(1, 625, .1, 25), (2, 1500, .1, 25), (3, 3000, .3, 25), (5, 4000, .1, 25), (3, 2000, .1, 9),
                                              (2, 900, 0.0, 36)])
@pytest.mark.parametrize("limited", [False, True])
def test_make_edges_bit_exact_vs_reference(q, n, missing, cell, limited):
    """tree_dep.cpp:75-130 (make_edges) and :133-186 (make_edges_limited) on the parent-child maps of real trees"""
    pb = common.make_problem(q, n, missing=missing, cell_size=cell)
    t, y = pb["tree"], pb["d"]["y"]
    ne = np.unique(t["blocking"][np.isfinite(y)])  # R/spamtree_fit.R:299-303
    r = ref.make_edges(t["parchi_map"], ne, t["res_is_ref"], limited)
    g = (sb.make_edges_limited if limited else sb.make_edges)(t["parchi_map"], ne, t["res_is_ref"])
    o = orc.make_edges(t["parchi_map"], ne, t["res_is_ref"], limited)
    for k in ("parents", "children"):
        assert _same_lists(r[k], g[k]), ("product", k)
        assert _same_lists(r[k], o[k]), ("oracle", k)
    if not limited:  # ... and they are what the tree builder handed to the model
        assert _same_lists(r["parents"], common.lists(t["parents_ptr"], t["parents_idx"]))
        assert _same_lists(r["children"], common.lists(t["children_ptr"], t["children_idx"]))


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_make_edges_random_maps_vs_reference(seed):
    """synthetic parent-child maps: ragged depth (NaN tails), a non-reference last level, some blocks empty"""
    rng = np.random.default_rng(seed)
    L = int(rng.integers(2, 6))
    rows, nxt = [], 1
    width = [1]
    for lev in range(1, L):
        width.append(width[-1] * int(rng.integers(2, 4)))
    ids = []
    for lev in range(L):
        ids.append(np.arange(nxt, nxt + width[lev]))
        nxt += width[lev]
    for leaf in range(width[-1]):
        chain, pos = [], leaf
        for lev in range(L - 1, -1, -1):
            chain.append(ids[lev][pos])
            if lev:
                pos = pos * width[lev - 1] // width[lev]
        chain = chain[::-1]
        cut = int(rng.integers(1, L + 1)) if rng.random() < .3 else L
        rows.append([float(c) if i < cut else np.nan for i, c in enumerate(chain)])
    pm = np.unique(np.array(rows), axis=0)
    pm = pm[np.lexsort(tuple(np.nan_to_num(pm[:, c], nan=1e9) for c in range(L - 1, -1, -1)))]
    # the reference sizes its lists by max(last column): make sure the largest id sits there
    pm[-1, :] = [float(ids[lev][-1]) for lev in range(L)]
    nb = int(np.nanmax(pm[:, -1]))
    ne = np.sort(rng.choice(np.arange(1, nb + 1), size=max(1, int(.8 * nb)), replace=False))
    rr = np.ones(L, dtype=np.int64)
    if rng.random() < .5:
        rr[-1] = 0
    for limited in (False, True):
        r = ref.make_edges(pm, ne, rr, limited)
        g = (sb.make_edges_limited if limited else sb.make_edges)(pm, ne, rr)
        o = orc.make_edges(pm, ne, rr, limited)
        for k in ("parents", "children"):
            assert _same_lists(r[k], g[k]), ("product", k, limited)
            assert _same_lists(r[k], o[k]), ("oracle", k, limited)


@pytest.mark.parametrize("n,d,k", [(1000, 2, (5, 5)), (257, 2, (10, 20)), (64, 3, (1, 2, 7)), (5, 2, (40, 40))])
def test_part_axis_parallel_lmt_bit_exact_vs_reference(n, d, k):
    """tree_dep.cpp:42-67, thresholds from kthresholds (:16-27) — incl. ties exactly at a threshold"""
    rng = np.random.default_rng(n)
    coords = np.round(rng.random((n, d)), 2)  # rounding produces ties with the thresholds
    thr = [ref.kthresholds(coords[:, j], k[j]) for j in range(d)]
    for j in range(d):
        assert np.array_equal(thr[j], sb.kthresholds(coords[:, j], k[j]))
        assert np.array_equal(thr[j], orc.kthresholds(coords[:, j], k[j]))
    r = ref.part_axis_parallel_lmt(coords, thr)
    assert np.array_equal(r, sb.part_axis_parallel_lmt(coords, thr))
    assert np.array_equal(r, orc.part_axis_parallel_lmt(coords, thr))


@pytest.mark.parametrize("npar", [4, 8, 15, 28])
def test_ramadapt_and_proposal_vs_reference(npar):
    """class RAMAdapt (mh_adapt.h:40-135), par_huvtransf_* (mh_adapt.cpp:3-15), unif_bounds (:188-202), calc_jacobian
    (:230-239), do_I_accept (:20-36) over a recorded (U, alpha) sequence: the product's host code = the reference's"""
    rng = np.random.default_rng(npar)
    steps = 180  # 50 warm-up iterations (g0), then the adaptive regime
    U = rng.standard_normal((steps, npar))
    alpha = np.where(rng.random(steps) < .2, 0.0, np.exp(rng.normal(-1, 2, steps)))  # incl. alpha = 0 (unacceptable) and > 1
    A = rng.standard_normal((npar, npar)) * .05
    sd0 = A @ A.T + np.eye(npar) * 1e-2
    pr, tr = ref.ram_adapt(sd0, U, alpha)
    pg, tg = sb.ram_adapt(sd0, U, alpha)
    assert relerr(pg, pr) <= 1e-12
    assert max(relerr(tg[i], tr[i]) for i in range(steps)) <= 1e-12
    q = {4: 1, 8: 2, 15: 3, 28: 5}[npar]
    bounds = synth.default_bounds(q)
    lo, hi = bounds[:, 0], bounds[:, 1]
    par = lo + (hi - lo) * rng.random(npar)
    assert relerr(sb.par_huvtransf_back(sb.par_huvtransf_fwd(par, bounds), bounds), par) <= 1e-12
    for i in range(0, steps, 7):
        scale = 1.0 if i % 21 else 400.0  # large steps run into the bounds (unif_bounds clips)
        nr, jr, obr = ref.propose(par, bounds, tr[i] * scale, U[i])
        ng, jg, obg = sb.mh_propose(par, bounds, tg[i] * scale, U[i])
        assert relerr(ng, nr) <= 1e-12 and obr == obg
        assert jg == jr or abs(jg - jr) <= 1e-12 * max(1.0, abs(jr))  # (a saturated logistic gives -inf in both)
    for la, u in [(-.5, .3), (-.5, .9), (.1, .999), (np.nan, .0001), (-np.inf, 1e-9), (np.inf, .5), (-1e-3, np.exp(-1e-3) - 1e-9)]:
        assert ref.do_i_accept(la, u) == sb.do_I_accept(la, u)
    with pytest.raises(sb.SpamTreeError):
        sb.ram_adapt(-np.eye(npar), U[:1], alpha[:1])  # not positive definite: the reference's arma::chol throws


CHAINS = [
    # q, n, missing, limited, sd, keep, burn, thin, adapting, predicts, tol
    (1, 625, .1, False, 1e-2, 15, 60, 2, True, True, 5e-9),    # the README shape; burn-in crosses into the adaptive regime (g0 = 50)
    (2, 900, .1, False, 1e-7, 65, 0, 1, True, True, 5e-9),     # every iteration saved, across g0
    (3, 1200, .2, False, 1e-7, 40, 0, 2, True, True, 5e-9),
    (3, 1000, .1, True, 1e-7, 28, 0, 1, False, False, 5e-9),   # limited tree, fixed proposal, no prediction
    (5, 1500, .1, False, 1e-7, 16, 0, 1, True, True, 5e-9),
]


@pytest.mark.parametrize("q,n,missing,limited,sd,keep,burn,thin,adapting,predicts,tol", CHAINS)
def test_oracle_chain_equals_the_references_own_driver(q, n, missing, limited, sd, keep, burn, thin, adapting, predicts, tol):
    """spamtree_mv_mcmc (spamtree_fit.cpp:5-430) compiled unmodified and run on the shared host stream vs the oracle's
    restatement of the loop: same accept decisions, theta / beta / tausq / paramsd / w / yhat of every saved iteration"""
    pb = common.make_problem(q, n, missing=missing, limited=limited)
    d, t = pb["d"], pb["tree"]
    bounds = synth.default_bounds(q)
    npar = pb["theta"].size
    msd = np.eye(npar) * sd
    r = ref.spamtree_mv_mcmc(d["y"], d["X"], d["coords"], d["mv_id"], t["res_is_ref"], pb["csr"], limited, t["block_names"],
                             t["block_groups"], pb["beta"], pb["theta"], pb["tausq"], bounds, msd, keep, burn, thin, adapting=adapting,
                             sample_predicts=predicts, seed=11)
    om = common.oracle_model(pb, flags=orc.FLAG_Q1_NORM_EXPANSION if q == 1 else 0)
    o = om.mcmc(bounds, msd, keep, burn, thin, adapting=adapting, sample_predicts=predicts, seed=11)
    assert np.array_equal(r["block_ct_obs"], om.geti("block_ct_obs"))
    plen = np.array([om.geti("parents_indexing", u).size for u in range(t["n_blocks"])])
    assert np.array_equal(r["parents_indexing_len"], plen)
    # the chain moved (some proposals accepted, some rejected) — otherwise the comparison says little
    assert 0 < o["n_accepted"] < keep * thin + burn
    if burn == 0:
        moved = np.any(np.diff(r["theta_mcmc"], axis=1) != 0, axis=0)
        assert moved.any() and not moved.all()
    for k in ("theta_mcmc", "tausq_mcmc", "beta_mcmc", "paramsd", "w_mcmc", "yhat_mcmc"):
        assert relerr(o[k], r[k]) <= tol, (k, relerr(o[k], r[k]))
    om.close()


@pytest.mark.parametrize("ncol", [1, 2])
def test_oracle_chain_with_one_or_two_regressors_vs_the_reference(ncol):
    """p = 1 (an intercept-only design, the commonest call of spamtree()) and p = 2 with q = 2: the beta step's p x p algebra
    (spamtree_model.cpp:1364-1391) at sizes where any layout that assumes p >= 3 goes wrong"""
    pb = common.make_problem(2, 900)
    d, t = pb["d"], pb["tree"]
    X = np.ascontiguousarray(d["X"][:, :ncol])
    pb["d"] = dict(d, X=X)
    pb["beta"] = np.zeros(ncol)
    bounds, npar = synth.default_bounds(2), pb["theta"].size
    msd = np.eye(npar) * 1e-7
    r = ref.spamtree_mv_mcmc(d["y"], X, d["coords"], d["mv_id"], t["res_is_ref"], pb["csr"], False, t["block_names"], t["block_groups"],
                             pb["beta"], pb["theta"], pb["tausq"], bounds, msd, 20, 0, 1, adapting=True, sample_predicts=True, seed=4)
    om = common.oracle_model(pb, flags=0)
    o = om.mcmc(bounds, msd, 20, 0, 1, adapting=True, sample_predicts=True, seed=4)
    assert r["beta_mcmc"].shape[0] == ncol
    for k in ("theta_mcmc", "tausq_mcmc", "beta_mcmc", "w_mcmc", "yhat_mcmc"):
        assert relerr(o[k], r[k]) <= 5e-9, (k, relerr(o[k], r[k]))
    om.close()
