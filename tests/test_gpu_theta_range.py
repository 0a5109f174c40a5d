"""The CUDA path across the theta box the sampler walks (tests/theta_range.py), against extended-precision truth: every
covariance entry against exp of the table in long double, BUILD (H, Ri, log-density, log-determinant), a Gibbs sweep with
shared z (w, Sigi_tot / Smu_tot probes), LLW, the integrated log-likelihood, predict_new, and the ok / not-positive-definite
decisions; the oracle alongside.  Where a point is beyond FP64 for the reference algorithm too, the bar is 4 x the oracle's
own distance from the truth (as in test_gpu_fullsize.py); every point prints cond(K_pa), both errors and the smallest
relative Cholesky pivot, so the printout shows where 1e-9 stops being attainable and why."""
import numpy as np
import pytest

import common
import iloo_ref
import launch_configs as lc
import spamtree_b200 as sb
import theta_range as tr
from common import orc, relerr
from spamtree_b200 import _lib, synth

pytestmark = pytest.mark.gpu
TOL = 1e-9
EPS = 2.0 ** -52

PROBLEMS = {
    "q1_n625": lambda: common.make_problem(1, 625),
    "q2_n1200_limited": lambda: common.make_problem(2, 1200, limited=True),
    "q3_n900": lambda: common.make_problem(3, 900),
    "q5_n2000": lambda: common.make_problem(5, 2000, missing=.15),
    "shape_ref_m_edges": lambda: lc.problem("shape_ref_m_edges"),   # reference blocks of m = 1 ... 118 (m > 32 included)
}
SUBSET = {"shape_ref_m_edges": ("start", "long", "var_hi", "random0", "random1")}
VISITED = {"q1_n625", "q3_n900"}   # points of a device chain run from the start of spamtree()


def _visited(pb, iters=300, n_points=4, seed=5):
    """four theta draws spread over a device chain of `iters` iterations from the start, default mcmcsd = .01"""
    q = pb["q"]
    b = synth.default_bounds(q)
    m = common.product_model(dict(pb, theta=b.mean(axis=1)), keep_H=False)
    try:
        r = m.mcmc(b, np.eye(b.shape[0]) * .01, iters, 0, 1, adapting=True, rng_mode=1, seed=seed, save_w=False, save_yhat=False)
    finally:
        m.close()
    cols = [iters * (k + 1) // n_points - 1 for k in range(n_points)]
    print(f"visited points (q = {q}): {r['n_accepted']} of {iters} accepted")
    return [(f"visited{k}", r["theta_mcmc"][:, c].copy(), tr.TAU_INV[k % 3]) for k, c in enumerate(cols)]


def _ldrel(a, b):
    b = np.asarray(b, dtype=np.longdouble)
    return float(np.max(np.abs(np.asarray(a, dtype=np.longdouble) - b)) / np.max(np.abs(b))) if b.size else 0.0


def _near(a, b):
    b = np.asarray(b, dtype=np.longdouble)
    return float(np.max(np.abs(np.asarray(a, dtype=np.longdouble) - b) / np.maximum(np.abs(b), 1)))


# ------------------------------------------------------------------------------------------------ covariance entries
@pytest.mark.parametrize("q", [2, 3, 5])
def test_covariance_entry_by_entry(q):
    """CrossCovarianceAG10 (the multivariate export: q >= 2) with r h swept over [0, 760] for every term of every table slot:
    exponents 0 up to ~1100 on the other term, h = 0 exactly, both sides of exp_neg's flush (e > 1000, r h ~ 693.8).
    Distances of 26 significant bits from a location at the origin make h and dx^2 exact, so the device's argument is
    fl(r h), the same product numpy forms; the truth is c1 exp(-fl(r1 h)) + c2 exp(-fl(r2 h)) in long double from the
    table of make_covtab_hd (tr.covtab, float64 by the same operations).  The bound is 4 units of 2^-52 of the two terms
    plus 2^-1000 (|c1| + |c2|): exp_neg returns 0 for exp(-a) below 2^-1000 instead of going on into the subnormals."""
    t = np.concatenate([[0.0], np.linspace(0, 760, 401)[1:], 693.8 + np.linspace(-3, 3, 61), [5e-7, 1e-6, 1e-3, 1.0]])
    worst = 0.0
    for name, th, _ in tr.points(q):
        ai1, ai2, phi, tm, D = (np.asarray(a, dtype=np.float64) for a in tr.theta_unpack(np.asarray(th), q))
        c1, r1, c2, r2 = tr.covtab(th, q)
        hs, mvb, slot_i = [], [], []
        for i in range(q):
            for j in range(q):
                for r in (r1[i, j], r2[i, j]):
                    if r > 0:
                        h = t / r
                        m, e = np.frexp(h)
                        h = np.ldexp(np.round(np.ldexp(m, 26)), e - 26)   # 26 significant bits: dx * dx is exact
                        hs.append(h)
                        mvb.append(np.full(h.size, j + 1))
                        slot_i.append(np.full(h.size, i))
        h, mvb, si = np.concatenate(hs), np.concatenate(mvb), np.concatenate(slot_i)
        xa, ma = np.zeros((q, 2)), np.arange(1, q + 1)
        xb = np.stack([h, np.zeros_like(h)], axis=1)
        C = sb.CrossCovarianceAG10(xa, ma, xb, mvb, ai1, ai2, phi, tm, D)   # q x nb
        got = C[si, np.arange(h.size)]
        i, j = si, mvb - 1
        ld = np.longdouble
        e1, e2 = np.exp(-(r1[i, j] * h).astype(ld)), np.exp(-(r2[i, j] * h).astype(ld))
        want = c1[i, j].astype(ld) * e1 + c2[i, j].astype(ld) * e2
        bound = 4 * EPS * (np.abs(c1[i, j]) * e1 + np.abs(c2[i, j]) * e2) + 2.0 ** -1000 * (np.abs(c1[i, j]) + np.abs(c2[i, j]))
        err = np.abs(got.astype(ld) - want)
        k = int(np.argmax(err / np.maximum(bound, 1e-300)))
        worst = max(worst, float(err[k] / bound[k]) if bound[k] > 0 else float(err[k] > 0) * np.inf)
        assert np.all(err <= bound), (name, float(h[k]), int(i[k]), int(j[k]), float(got[k]), float(want[k]), float(bound[k]))
        assert np.all(got[h == 0] == (c1[i, j] + c2[i, j])[h == 0])
    print(f"q = {q}: {len(tr.points(q))} points, worst error / bound {worst:.3f}")


# ------------------------------------------------------------------------------------------------ one point of a problem
def _keep_loglik_int(m):
    m._chk(_lib.lib.st_keep_samples_on_device(m._h, _lib.ST_KEEP_LOGLIK_INT))


def _run_point(pb, prob, name, theta, tau_inv, fails, rng):
    q, n = pb["q"], pb["n"]
    d = pb["d"]
    y = d["y"]
    obs_rows = np.isfinite(y)
    tau = np.full(q, tau_inv)
    line = {"cond": np.nan, "margin": np.nan}

    def check(ok, what):
        if not ok:
            fails.append(f"{prob} {name}: {what}")

    gm, om = common.product_model(pb, keep_H=True), common.oracle_model(pb)   # built at the parity point; theta as a proposal
    try:
        w0 = rng.standard_normal(n) * .5
        for m in (gm, om):
            m.w = w0
            m.set_tausq_inv(tau)
            assert m.get_loglik_comps_w(0)[0] and m.get_loglik_comps_w(1)[0]
        ll_before = gm.get_loglik_comps_w(1)[1]
        for m in (gm, om):
            m.theta_update(1, theta)
        okg, llg, ldg = gm.get_loglik_comps_w(1)
        oko, llo, ldo = om.get_loglik_comps_w(1)
        tw, bl = tr.ld_blocks(pb, theta)
        margin = min(min(b.margin_pa, b.margin_R) for b in bl.values())
        cond = max(b.cond_pa for b in bl.values())
        line.update(cond=cond, margin=margin, ok=f"{int(okg)}/{int(oko)}")
        # ---- decisions
        if margin > 1e-10:
            check(okg, f"BUILD refused a theta with every pivot margin above 1e-10 ({margin:.2e})")
        if okg != oko:
            print(f"  {prob} {name}: ok GPU {okg} oracle {oko} at margin {margin:.2e}")
            check(margin < 1e-12, f"ok differs from the oracle's at margin {margin:.2e}")
        if not okg:
            check(llg == ll_before, "a refused BUILD changed the slot's log-density")
            check(np.all(np.isfinite(gm.w)), "NaN in w after a refused BUILD")
            gm.theta_update(1, pb["theta"])
            check(gm.get_loglik_comps_w(1)[0], "the slot does not recover after a refused BUILD")
            return line
        for m in (gm, om):
            m.accept_make_change()
        # ---- BUILD against the truth, the oracle alongside
        eg, eo = {"H": 0.0, "Ri": 0.0}, {"H": 0.0, "Ri": 0.0}
        for u, b in bl.items():
            if b.Ri is None:
                continue
            mu = tw.rows[u].size
            if tw.prow(u).size:
                eg["H"] = max(eg["H"], _ldrel(gm.node_state("H", u).reshape(-1, mu).T, b.H))
                if oko:
                    eo["H"] = max(eo["H"], _ldrel(om.get("H", u).reshape(-1, mu).T, b.H))
            Rg = gm.node_state("Ri", u)
            Ro = (om.get("Ri", u) if tw.isref[u] else om.get("ccholprecdiag", u)) if oko else None
            if tw.isref[u]:
                Rg = Rg.reshape(mu, mu).T
                Ro = None if Ro is None else Ro.reshape(mu, mu).T
            eg["Ri"] = max(eg["Ri"], _ldrel(Rg, b.Ri))
            if oko:
                eo["Ri"] = max(eo["Ri"], _ldrel(Ro, b.Ri))
        lt, dt = tr.ld_loglik(pb, theta, w0, (tw, bl))
        eg["ll"], eg["ld"] = abs(llg - lt) / abs(lt), abs(ldg - dt) / max(abs(dt), 1.0)
        eo["ll"], eo["ld"] = abs(llo - lt) / abs(lt), abs(ldo - dt) / max(abs(dt), 1.0)
        line.update(eg=max(eg.values()), eo=max(eo.values()) if oko else np.nan)
        if not oko:
            return line
        slack = max(TOL, 4 * max(eo.values()))
        line["slack"] = slack
        for k in eg:
            check(eg[k] <= slack, f"BUILD {k}: {eg[k]:.2e} from the truth, bar {slack:.2e} (oracle {eo[k]:.2e})")
        check(abs(llg - llo) <= 2 * slack * abs(llo), f"loglik differs from the oracle's by {abs(llg - llo) / abs(llo):.2e}")
        # ---- Gibbs with shared z
        z = rng.standard_normal(n)
        iloo = pb.get("limited", False)
        if iloo:
            _keep_loglik_int(gm)
        errs = []
        for m, exc in ((gm, sb.SpamTreeError), (om, RuntimeError)):
            try:
                m.deal_with_w(z)
                errs.append(None)
            except exc as ex:
                errs.append(ex)
        if margin > 1e-10:
            check(errs[0] is None, f"the sweep failed at margin {margin:.2e}: {errs[0]}")
        if (errs[0] is None) != (errs[1] is None):
            print(f"  {prob} {name}: sweep GPU {errs[0]} oracle {errs[1]} at margin {margin:.2e}")
            check(margin < 1e-12, "the sweep's decision differs from the oracle's")
        if errs[0] is not None or errs[1] is not None:
            return line
        # against the same sweep in long double: the oracle's distance from it (its BUILD error carried through the
        # block and its children) sets the bar, as for BUILD; the GPU - oracle distance is printed
        w1 = gm.w
        tq_row = tau[d["mv_id"] - 1]
        resid = np.where(obs_rows, y, 0.0) - gm.params()["XB"]
        wt, pt = tr.ld_gibbs_sweep(pb, theta, w0, z, tq_row, resid, (tw, bl))
        gs = {"w": _ldrel(w1[obs_rows], wt[obs_rows]), "Sigi_tot": 0.0, "Smu_tot": 0.0}
        go = {"w": _ldrel(om.w[obs_rows], wt[obs_rows]), "Sigi_tot": 0.0, "Smu_tot": 0.0}
        for u, (St, Mt) in pt.items():
            for k, t in (("Sigi_tot", St.ravel()), ("Smu_tot", Mt)):
                gs[k] = max(gs[k], _ldrel(gm.node_state(k, u), t))
                go[k] = max(go[k], _ldrel(om.get(k, u), t))
        gslack = max(slack, 4 * max(go.values()))
        ew = relerr(w1[obs_rows], om.w[obs_rows])
        es = max(relerr(gm.node_state("Sigi_tot", u), om.get("Sigi_tot", u)) for u in bl)
        em = max(relerr(gm.node_state("Smu_tot", u), om.get("Smu_tot", u)) for u in bl)
        line.update(w=ew, sig=es, smu=em, gibbs_g=max(gs.values()), gibbs_o=max(go.values()))
        for k in gs:
            check(gs[k] <= gslack, f"Gibbs {k}: {gs[k]:.2e} from the truth, bar {gslack:.2e} (oracle {go[k]:.2e})")
        # ---- integrated log-likelihood (limited tree: the dense prior conditional is what the sweep conditions on)
        if iloo:
            got = gm.loglik_int()
            tq = tq_row
            Q = tr.ld_dense_precision(pb, theta, (tw, bl))
            rows, truth, blk, qd = [], [], [], []
            for u in bl:
                ru = tw.rows[u]
                below = iloo_ref._rows_at_or_below(tw, tw.level[u])
                state = np.asarray(w0, dtype=np.longdouble)
                state[below] = w1[below]
                o = ru[obs_rows[ru]]
                if not o.size:
                    continue
                Sig, Smu = gm.node_state("Sigi_tot", u), gm.node_state("Smu_tot", u)
                if tw.isref[u]:
                    Sig = Sig.reshape(ru.size, ru.size)
                keep = obs_rows[ru]
                blk.append(iloo_ref.block_terms(Sig, Smu, w1[ru], z[ru], tq[ru], resid[ru])[keep])
                truth.append(iloo_ref.dense_terms(Q, state, o, tq[o], resid[o]))
                qd.append(np.diag(Q)[o].astype(np.float64))
                rows.append(o)
            rows, truth, blk, qd = (np.concatenate(a) for a in (rows, truth, blk, qd))
            ek, eb = _near(got[rows], truth), _near(blk, truth)
            est = tq[rows] / qd * EPS      # the cancellation of Sigi_tot_aa - tausq_inv, relative to Q'_aa
            line.update(iloo=ek, iloo_blk=eb)
            check(ek <= 1e-8, f"integrated log-likelihood {ek:.2e} from the truth")
            if name == "var_hi" and q >= 2:
                print(f"  {prob} var_hi: cancellation estimate tausq_inv / Q'_aa 2^-52: median {np.median(est):.2e}, "
                      f"above 1e-7 on {np.mean(est > 1e-7):.0%} of the rows; error of the kernel {ek:.2e}, of "
                      f"Sigi_tot_aa - tausq_inv {eb:.2e}")
                check(np.mean(est > 1e-7) > .5, "var_hi does not reach the cancellation")
                check(ek <= .1 * eb, f"integrated log-likelihood at var_hi: {ek:.2e} against {eb:.2e} of Sigi_tot_aa - tausq_inv")
        # ---- LLW at the new w against a fresh BUILD
        lg = gm.get_loglik_w(0)[0]
        okb, lb, _ = gm.get_loglik_comps_w(0)
        check(okb and abs(lg - lb) <= 1e-10 * abs(lb), f"LLW {lg!r} against BUILD {lb!r}")
        # ---- prediction at new locations from this theta and w
        if "indexing_ptr" in pb["tree"] and not prob.startswith("shape_"):
            obs_at = np.flatnonzero(obs_rows)[:4]
            cn = np.vstack([rng.random((120, 2)) * 1.2 - .1, d["coords"][obs_at]])   # a few on observed locations
            mvn = np.r_[rng.integers(1, q + 1, 120), d["mv_id"][obs_at]]
            tn = sb.make_tree(d["coords"], y, d["mv_id"], cell_size=25, seed=0, coords_new=cn, mv_id_new=mvn,
                              limited_tree=pb["limited"])["new"]
            mt, vt, kii, pmarg = tr.ld_predict(pb, theta, tn, cn, mvn, w1)
            m64, v64, _, _ = tr.ld_predict(pb, theta, tn, cn, mvn, w1, dtype=np.float64)
            samples = {"theta_mcmc": theta[:, None], "beta_mcmc": np.zeros((3, 1, q)), "tausq_mcmc": np.full((q, 1), 1 / tau_inv),
                       "w_mcmc": w1[:, None]}
            try:
                out = gm.predict_new(cn, None, mvn, tn, samples, moments=True)
            except sb.SpamTreeError as ex:
                check(ex.code == 3 and pmarg <= 1e-10, f"predict_new refused at margin {pmarg:.2e}: {ex}")
                return line
            mg, sg = out["mean"][:, 0], out["sd"][:, 0]
            vg = sg ** 2
            mbar = max(TOL * float(np.max(np.abs(mt))), 4 * float(np.max(np.abs(m64 - mt))))
            emean = float(np.max(np.abs(mg - mt)))
            well = vt > 1e-6 * kii
            rel_slack = max(TOL, 4 * float(np.max(np.abs(v64 - vt)[well] / vt[well]))) if well.any() else TOL
            ev = float(np.max(np.abs(vg - vt)[well] / vt[well])) if well.any() else 0.0
            abs_bar = max(4 * float(np.max(np.abs(v64 - vt)[~well])) if (~well).any() else 0.0, 4 * EPS * float(np.max(kii)))
            evs = float(np.max(np.abs(vg - vt)[~well])) if (~well).any() else 0.0
            line.update(pred_mean=emean / float(np.max(np.abs(mt))), pred_var=ev)
            check(emean <= mbar, f"predict mean {emean:.2e} from the truth, bar {mbar:.2e}")
            check(ev <= rel_slack, f"predict var {ev:.2e} relative where the Schur complement > 1e-6 K_ii, bar {rel_slack:.2e}")
            check(evs <= abs_bar, f"predict var {evs:.2e} absolute on small Schur complements, bar {abs_bar:.2e}")
            check(np.all(vt[sg == 0] <= abs_bar), "sd = 0 where the Schur complement is positive")
            check(np.all(np.isfinite(mg)) and np.all(sg >= 0), "predict_new: non-finite mean or negative sd")
        return line
    finally:
        gm.close()
        om.close()


@pytest.mark.parametrize("prob", list(PROBLEMS))
def test_theta_range(prob):
    pb = PROBLEMS[prob]()
    q = pb["q"]
    pts = tr.points(q)
    if prob in SUBSET:
        pts = [p for p in pts if p[0] in SUBSET[prob]]
    if prob in VISITED:
        pts = pts + _visited(pb)
    rng = np.random.default_rng(11)
    fails = []
    print(f"\n{prob} (q = {q}, n = {pb['n']}): point  tausq_inv  ok(GPU/oracle)  cond(K_pa)  margin  BUILD err GPU / oracle  "
          f"bar  | GPU-oracle w  Sigi  Smu | sweep err GPU / oracle | iloo (blk) | predict mean  var")
    for name, th, tau in pts:
        ln = _run_point(pb, prob, name, th, tau, fails, rng)
        f = lambda k: f"{ln[k]:.1e}" if k in ln and np.isfinite(ln[k]) else "-"
        print(f"  {name:9s} {tau:7.0e}  {ln.get('ok', '-'):4s} {f('cond')} {f('margin')}  {f('eg')} / {f('eo')}  {f('slack')} | "
              f"{f('w')} {f('sig')} {f('smu')} | {f('gibbs_g')} / {f('gibbs_o')} | {f('iloo')} ({f('iloo_blk')}) | {f('pred_mean')} {f('pred_var')}", flush=True)
    assert not fails, "\n".join(fails)


def test_entry_point_at_its_own_start():
    """spamtree() from the middle of the box, q = 3: the saved thetas stay in the box and every output is finite except
    the NaN rows the API documents (the per-row criteria where y is missing)"""
    d = synth.make_data(3, 900, seed=2021)
    r = sb.spamtree(d["y"], d["X"], d["coords"], d["mv_id"], mcmc={"keep": 50, "burn": 0, "thin": 1}, seed=1, loo_integrated=True)
    b = synth.default_bounds(3)
    th = r["theta_mcmc"]
    assert th.shape == (b.shape[0], 50)
    assert np.all(th >= b[:, :1]) and np.all(th <= b[:, 1:])
    for k in ("w_mcmc", "yhat_mcmc", "beta_mcmc", "tausq_mcmc", "paramsd"):
        assert np.all(np.isfinite(r[k])), k
    miss = np.isnan(d["y"][r["coordsinfo"]["ix"] - 1])
    ci = r["fit_criteria_integrated"]
    for k, v in ci.items():
        v = np.asarray(v, dtype=np.float64)
        if v.ndim == 1 and v.size == miss.size:
            assert np.all(np.isnan(v[miss])) and np.all(np.isfinite(v[~miss])), k
        elif k not in ("dbar", "dhat", "p_dic", "dic"):   # (the DIC totals of the integrated criteria are NaN)
            assert np.all(np.isfinite(v)), k
    print(f"spamtree q = 3, n = 900, 50 iterations from the start: n_accepted {r['n_accepted']}, n_chol_fail {r['n_chol_fail']}")
