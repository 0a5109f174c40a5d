"""The points and extended-precision references of tests/theta_range.py against independent statements: the start of
spamtree(), dense_twin.Twin at the parity points, mpmath at 50 digits, conditioning of the dense joint normal, and the
monotonicity of the pivot margins in the decay."""
import math

import mpmath
import numpy as np
import pytest

import common
import iloo_ref
import theta_range as tr
from dense_twin import Twin, block_truth_ld, cov
from spamtree_b200 import synth

QS = [1, 2, 3, 5]


class _Started(Exception):
    pass


@pytest.mark.parametrize("q", QS)
def test_start_is_the_start_of_spamtree(q, monkeypatch):
    import spamtree_b200.api as api
    seen = {}

    def capture(*a, **kw):  # the handle spamtree() opens for its chain: record theta, open nothing
        seen["theta"] = np.asarray(a[12], dtype=np.float64).copy()
        raise _Started

    monkeypatch.setattr(api, "SpamTreeMV", capture)
    d = synth.make_data(q, 200, seed=3)
    with pytest.raises(_Started):
        api.spamtree(d["y"], d["X"], d["coords"], d["mv_id"], mcmc={"keep": 2})
    pts = {name: th for name, th, _ in tr.points(q)}
    assert np.array_equal(pts["start"], seen["theta"])


@pytest.mark.parametrize("q", QS)
def test_points_lie_in_the_box(q):
    b = synth.default_bounds(q)
    pts = tr.points(q)
    names = [p[0] for p in pts]
    assert len(set(names)) == len(names) and sum(n.startswith("random") for n in names) == 8
    for name, th, tau in pts:
        assert th.shape == (b.shape[0],) and np.all(th >= b[:, 0]) and np.all(th <= b[:, 1]), name
        assert tau in tr.TAU_INV
    assert {tau for _, _, tau in pts} == set(tr.TAU_INV)
    assert dict((n, t) for n, _, t in pts)["var_hi"] == 1e3  # the cancellation point of the integrated log-likelihood
    # the random points spread over the box: each parameter reaches both halves of its range
    R = np.array([th for n, th, _ in pts if n.startswith("random")])
    mid = b.mean(axis=1)
    assert np.all((R < mid).any(axis=0) & (R > mid).any(axis=0))


def test_covtab_is_the_covariance():
    """the float64 table reproduces dense_twin.cov (the formulas of covariance_functions.cpp) to rounding"""
    rng = np.random.default_rng(1)
    for q in (1, 2, 3, 5):
        for name, th, _ in tr.points(q):
            c1, r1, c2, r2 = tr.covtab(th, q)
            xa, xb = rng.random((6, 2)), rng.random((7, 2))
            ma, mb = rng.integers(1, q + 1, 6), rng.integers(1, q + 1, 7)
            h = np.sqrt(((xa[:, None] - xb[None]) ** 2).sum(-1))
            i, j = ma[:, None] - 1, mb[None, :] - 1
            got = c1[i, j] * np.exp(-r1[i, j] * h) + c2[i, j] * np.exp(-r2[i, j] * h)
            want = cov(xa, ma, xb, mb, th, q)
            assert np.allclose(got, want, rtol=1e-12, atol=1e-300), (q, name)


def _mp_cov(xa, ma, xb, mb, theta, q):
    """dense_twin.cov's formula at 50 significant digits from the same float64 inputs"""
    mpmath.mp.dps = 50
    th = [mpmath.mpf(float(x)) for x in theta]
    ai1, ai2, phi = th[:q], th[q:2 * q], th[2 * q:3 * q]
    ncb = 3 if q > 2 else 1
    tm = th[3 * q:3 * q + ncb]
    D = [[mpmath.mpf(0)] * q for _ in range(q)]
    ix = 3 * q + ncb
    for j in range(q):
        for i in range(j + 1, q):
            D[i][j] = D[j][i] = th[ix]
            ix += 1
    out = []
    for a in range(len(xa)):
        for b in range(len(xb)):
            h = mpmath.sqrt(sum((mpmath.mpf(float(xa[a, k])) - mpmath.mpf(float(xb[b, k]))) ** 2 for k in range(2)))
            if q == 1:
                out.append(ai1[0] * mpmath.exp(-tm[0] * h))
                continue
            i, j = int(ma[a]) - 1, int(mb[b]) - 1
            v = D[i][j]
            if q > 2:
                psi = (1 + tm[0] * v) ** tm[1]
                base = mpmath.exp(-tm[2] * h / mpmath.sqrt(psi)) / psi
            else:
                base = mpmath.exp(-tm[0] * h / mpmath.sqrt(v + 1)) / (v + 1)
            out.append(ai1[i] ** 2 * base + ai2[i] ** 2 * mpmath.exp(-phi[i] * h) if v == 0 else ai1[i] * ai1[j] * base)
    return out


def test_long_double_covariance_against_mpmath():
    """300+ entries over the box: long double agrees with 50 digits to a few units of its own rounding, which grows with
    the exponent r h (the argument is rounded before exp is taken)"""
    rng = np.random.default_rng(2)
    n_checked, worst = 0, 0.0
    for q in (1, 2, 3):
        for name, th, _ in tr.points(q):
            xa, xb = rng.random((3, 2)), rng.random((5, 2))
            ma, mb = rng.integers(1, q + 1, 3), rng.integers(1, q + 1, 5)
            got = cov(xa, ma, xb, mb, th, q, np.longdouble).ravel()
            want = _mp_cov(xa, ma, xb, mb, th, q)
            c1, r1, c2, r2 = tr.covtab(th, q)
            h = np.sqrt(((xa[:, None] - xb[None]) ** 2).sum(-1))
            i, j = ma[:, None] - 1, mb[None, :] - 1
            expo = np.maximum(r1[i, j], r2[i, j]).ravel() * h.ravel()   # the largest exponent of each entry
            for k, wv in enumerate(want):
                if wv == 0:
                    assert got[k] == 0
                    continue
                rel = float(abs(mpmath.mpf(str(got[k])) - wv) / abs(wv))  # (str: every digit of the long double)
                worst = max(worst, rel / (1 + expo[k]))
                assert rel <= 64 * 2.0 ** -64 * (1 + expo[k]), (q, name, k, rel, expo[k])
                n_checked += 1
    assert n_checked >= 300
    print(f"{n_checked} entries, worst long-double error / (1 + r h) {worst:.2e}")


@pytest.mark.parametrize("q,n", [(1, 300), (2, 400), (3, 450), (5, 600)])
def test_ld_loglik_equals_twin_at_the_parity_points(q, n):
    pb = common.make_problem(q, n)
    w = np.random.default_rng(4).standard_normal(n) * .5
    ll, ld = tr.ld_loglik(pb, pb["theta"], w)
    tw = Twin(pb)
    Q, logdet = tw.precision()
    assert abs(ld - logdet) <= 1e-12 * abs(logdet)
    assert abs(ll - tw.loglik(w)) <= 1e-12 * abs(ll)
    # ld_block is block_truth_ld (same algorithm, same numbers) plus the margins
    _, bl = tr.ld_blocks(pb, pb["theta"])
    u = max(bl, key=lambda u: tw.prow(u).size)
    H, Ri = block_truth_ld(tw.coords, tw.mv, tw.rows[u], tw.prow(u), pb["theta"], q, bool(tw.isref[u]))
    assert np.array_equal(H, bl[u].H) and np.array_equal(Ri, bl[u].Ri)
    assert all(0 < b.margin_pa <= 1 and 0 < b.margin_R <= 1 for b in bl.values())
    # the long-double precision is Twin's
    Qld = tr.ld_dense_precision(pb, pb["theta"], (tw, bl))
    assert np.max(np.abs(Qld - Q)) <= 1e-9 * np.max(np.abs(Q))


def test_dense_terms_on_the_ld_precision_is_conditioning():
    """iloo_ref.dense_terms on the long-double Q: w_a given the rest of w, N(w_a - (Q w)_a / Q_aa, 1 / Q_aa), equals
    conditioning the joint normal N(0, Q^-1) of the observed blocks' rows on the others (brute_loo's way)"""
    pb = common.make_problem(1, 300, limited=True)
    th = pb["theta"]
    tw, bl = tr.ld_blocks(pb, th)
    Q = tr.ld_dense_precision(pb, th, (tw, bl))
    B = np.concatenate([tw.rows[u] for u in bl])
    rng = np.random.default_rng(6)
    state = rng.standard_normal(tw.y.size)
    tq = np.full(tw.y.size, 4.0)
    resid = rng.standard_normal(tw.y.size)
    rows = B[:: 7]
    got = iloo_ref.dense_terms(Q, state.astype(np.longdouble), rows, tq[rows], resid[rows])
    S = np.linalg.inv(Q[np.ix_(B, B)].astype(np.float64))
    pos = {r: k for k, r in enumerate(B)}
    for a, g in zip(rows, got):
        i = pos[a]
        o = np.arange(B.size) != i
        k = S[i, o]
        sol = np.linalg.solve(S[np.ix_(o, o)], np.stack([state[B][o], k], axis=1))
        mean, var = k @ sol[:, 0], S[i, i] - k @ sol[:, 1]
        want = iloo_ref.norm_logpdf(resid[a], mean, var + 1 / tq[a])
        assert abs(float(g) - want) <= 1e-8 * max(1.0, abs(want)), (a, float(g), want)


def test_pivot_margins_are_monotone_in_the_decay():
    """on one fixed block with parents, both margins shrink as the range grows (decay from 1e3 to 1e-3): the block gets
    closer to singular; at 1e3 K is nearly diagonal and both are near 1"""
    pb = common.make_problem(1, 625)
    tw = Twin(pb)
    u = max((u for u in range(tw.nb) if tw.obs[u] and tw.isref[u]), key=lambda u: tw.prow(u).size)
    ms = []
    for phi in (1e3, 1e2, 10.0, 1.0, 1e-1, 1e-2, 1e-3):
        th = pb["theta"].copy()
        th[3] = phi
        b = tr.ld_block(tw.coords, tw.mv, tw.rows[u], tw.prow(u), th, 1, True)
        ms.append((b.margin_pa, b.margin_R))
    ms = np.array(ms)
    assert np.all(ms[0] > .9), ms
    assert np.all(np.diff(ms, axis=0) <= 0), ms
    assert ms[-1, 0] < 1e-2 and ms[-1, 1] < 1e-2, ms


def test_ld_predict_agrees_with_float64_at_a_parity_point():
    import spamtree_b200 as sb
    pb = common.make_problem(2, 600)
    d = pb["d"]
    rng = np.random.default_rng(8)
    cn = rng.random((80, 2))
    mvn = rng.integers(1, 3, 80)
    tn = sb.make_tree(d["coords"], d["y"], d["mv_id"], cell_size=25, seed=0, coords_new=cn, mv_id_new=mvn)["new"]
    w = rng.standard_normal(pb["n"])
    m1, v1, k1, mg = tr.ld_predict(pb, pb["theta"], tn, cn, mvn, w)
    m2, v2, k2, _ = tr.ld_predict(pb, pb["theta"], tn, cn, mvn, w, dtype=np.float64)
    assert 0 < mg <= 1 and np.all(v1 > 0) and np.all(v1 <= k1)
    assert np.max(np.abs(m2 - m1)) <= 1e-11 * np.max(np.abs(m1)) and np.max(np.abs(v2 - v1)) <= 1e-11 * np.max(k1)


@pytest.mark.parametrize("q,n,limited", [(1, 300, False), (3, 450, False), (2, 400, True)])
def test_ld_gibbs_sweep_is_twins_sweep(q, n, limited):
    pb = common.make_problem(q, n, limited=limited)
    rng = np.random.default_rng(9)
    w0, z, resid = rng.standard_normal(n) * .5, rng.standard_normal(n), rng.standard_normal(n)
    tq = np.linspace(3, 8, q)[pb["d"]["mv_id"] - 1]
    tw = Twin(pb)
    w_tw, p_tw = tw.gibbs_sweep(w0, z, tq, resid)
    w_ld, p_ld = tr.ld_gibbs_sweep(pb, pb["theta"], w0, z, tq, resid)
    obs = np.concatenate([tw.rows[u] for u in p_ld])
    assert set(p_ld) == set(p_tw)
    assert common.relerr(w_ld[obs].astype(np.float64), w_tw[obs]) <= 1e-10
    for u in p_ld:
        for a, b in zip(p_ld[u], p_tw[u]):
            assert common.relerr(a.astype(np.float64), b) <= 1e-10, u
