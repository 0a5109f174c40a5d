"""tests/iloo_ref.py without a GPU: the integrated log-likelihood formed from what a Gibbs sweep has when it draws a block
(dense_twin.Twin.gibbs_sweep's probes, the block's new w and its normals) is the log-density of y_i - x_i'beta under the
prior conditional of w_i given the rest of w at that point of the sweep, plus tausq, on trees whose messages are current
(two-level and limited trees); and the closed-form leave-one-out predictive of the Gaussian model is the conditional of the
joint normal."""
import numpy as np
import pytest

import common
import iloo_ref
import spamtree_b200 as sb
from dense_twin import Twin
from spamtree_b200 import synth


def _two_level(q, n, cell_size=25):
    """a reference root and one level of non-reference blocks under it (and the prediction blocks of the missing rows)"""
    d = synth.make_data(q, n, missing=0.1, seed=2021)
    tree = sb.make_tree(d["coords"], d["y"], d["mv_id"], cell_size=cell_size, tree_depth=1)
    csr = (tree["indexing_ptr"], tree["indexing_idx"], tree["parents_ptr"], tree["parents_idx"], tree["children_ptr"],
           tree["children_idx"])
    return {"d": d, "tree": tree, "csr": csr, "theta": synth.theta_for(q), "beta": np.zeros(3), "tausq": 0.1, "q": q, "n": n,
            "limited": False}


PROBLEMS = {
    "two_level_q1": lambda: _two_level(1, 300),
    "two_level_q3_m40": lambda: _two_level(3, 450, cell_size=40),
    "limited_q1": lambda: common.make_problem(1, 400, limited=True),
    "limited_q2": lambda: common.make_problem(2, 500, limited=True),
}


def _sweep(pb, seed=3):
    tw = Twin(pb)
    rng = np.random.default_rng(seed)
    n, q = pb["n"], pb["q"]
    tau = np.array([3.0, 5.0, 8.0])[:q][pb["d"]["mv_id"] - 1]
    resid = np.where(np.isfinite(pb["d"]["y"]), pb["d"]["y"], 0.0) - 0.2
    w0 = rng.standard_normal(n) * .5
    z = rng.standard_normal(n)
    w1, probes = tw.gibbs_sweep(w0, z, tau, resid)
    return tw, w0, w1, z, tau, resid, probes


@pytest.mark.parametrize("name", sorted(PROBLEMS))
def test_sweep_formula_is_the_prior_conditional(name):
    pb = PROBLEMS[name]()
    tw, w0, w1, z, tau, resid, probes = _sweep(pb)
    assert any(tw.isref[u] for u in probes) and any(not tw.isref[u] for u in probes)
    rows, a, b = iloo_ref.sweep_terms(tw, w0, w1, z, tau, resid, probes)
    assert rows.size == np.unique(rows).size
    assert np.all(np.isfinite(a))
    assert np.max(np.abs(a - b) / np.maximum(np.abs(b), 1.0)) < 1e-9


def test_a_deeper_full_tree_has_stale_messages():
    """(the caveat of DESIGN.md §5f: a block's message to an ancestor other than its parent is formed before the blocks in
    between are drawn, so the reference blocks of a deeper full tree condition on a state the sweep never holds at once)"""
    pb = common.make_problem(1, 900)
    tw, w0, w1, z, tau, resid, probes = _sweep(pb)
    assert max(len(tw.parents[u]) for u in probes) >= 2
    rows, a, b = iloo_ref.sweep_terms(tw, w0, w1, z, tau, resid, probes)
    nonref = np.concatenate([tw.rows[u] for u in probes if not tw.isref[u]])
    keep = np.isin(rows, nonref)
    assert np.max(np.abs(a[keep] - b[keep])) < 1e-9  # rows of non-reference blocks take no messages
    assert np.max(np.abs(a[~keep] - b[~keep])) > 1e-6


@pytest.mark.parametrize("limited", [False, True])
def test_closed_form_loo_is_the_conditional(limited):
    pb = common.make_problem(1, 300, limited=limited)
    tw = Twin(pb)
    Q, _ = tw.precision()
    B = np.concatenate([tw.rows[u] for u in range(tw.nb) if tw.obs[u] > 0])
    y = pb["d"]["y"][B]
    obs = np.flatnonzero(np.isfinite(y))
    xb = 0.3 * np.ones(B.size)
    tausq = np.full(B.size, 0.05)
    mean, var, ll = iloo_ref.exact_loo(Q[np.ix_(B, B)], obs, y, xb, tausq)
    for i in (0, 7, obs.size // 2, obs.size - 1):
        m, v = iloo_ref.brute_loo(Q[np.ix_(B, B)], obs, y, xb, tausq, i)
        assert abs(mean[i] - m) <= 1e-8 * max(1.0, abs(m)) and abs(var[i] - v) <= 1e-8 * v
    assert np.all(np.isfinite(ll))
