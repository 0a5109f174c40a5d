"""Generates tests/golden/ref_*.npz by running THE REFERENCE'S OWN CODE: oracle/_ref/libspamtree_ref.so is the reference's
model layer (spamtree_model.cpp, covariance_functions.cpp, tree_utils.cpp, tree_dep.cpp, mh_adapt.cpp) compiled
unmodified from the reference package's src/ directory against the Armadillo/Rcpp stand-in of oracle/refshim/
(`make -C oracle ref`).  The reference's sources are not part of this repository, so its outputs are committed here as
fixtures; the CPU oracle and the CUDA path are both checked against them (tests/test_golden_reference.py).  The ref_chain_*.npz files are whole chains of the reference's own MCMC driver
(spamtree_fit.cpp, compiled unmodified as well).
Run (the reference's src/ is SPAMTREE_REF_SRC, else src/ under BASELINE.json's reference_path):
    python tests/golden/make_golden_from_reference.py"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import common  # noqa: E402
from oracle import ref  # noqa: E402

CASES = [(1, 625, False), (3, 900, False), (2, 1200, False), (3, 1100, True)]   # (q, n, limited_tree): README shape, q = 3, q = 2, a limited tree


def one(q, n, limited):
    pb = common.make_problem(q, n, limited=limited)
    d, t = pb["d"], pb["tree"]
    rm = ref.RefModel(d["y"], d["X"], d["coords"], d["mv_id"], t["res_is_ref"], pb["csr"], limited, t["block_names"], t["block_groups"],
                      pb["beta"], pb["theta"], pb["tausq"])
    rng = np.random.default_rng(100 + q)
    out = {"q": q, "n": n, "limited": int(limited), "blocking": t["blocking"], "theta": pb["theta"]}
    nb = t["n_blocks"]
    # ---- integer bookkeeping of the constructor (spamtree_model.cpp:194-420)
    for name in ["blocks_not_empty", "blocks_predicting", "block_is_reference", "block_ct_obs"]:
        out["i_" + name] = rm.geti(name)
    for name in ["parents_indexing", "children_indexing", "dim_by_parent", "this_is_jth_child"]:
        parts = [rm.geti(name, u) for u in range(nb)]
        out["i_" + name + "_ptr"] = np.cumsum([0] + [p.size for p in parts])
        out["i_" + name] = np.concatenate(parts) if parts else np.zeros(0, np.int64)
    # ---- BUILD at theta with a given w (get_loglik_comps_w_std :834-998)
    w0 = rng.standard_normal(n) * .5
    rm.w = w0
    ok, ll, ld = rm.get_loglik_comps_w(0)
    assert ok
    out.update(w0=w0, loglik=ll, logdet=ld, logdetCi_comps=rm.get("logdetCi_comps"))
    obs, isref = out["i_block_ct_obs"], out["i_block_is_reference"]
    npar = np.diff(t["parents_ptr"])
    for u in range(nb):
        if obs[u] == 0:
            continue
        if npar[u]:
            out[f"H_{u}"] = rm.get("H", u)                      # m x P, column-major
        out[f"Ri_{u}"] = rm.get("Ri", u) if isref[u] else rm.get("ccholprecdiag", u)
    # ---- GIBBS sweeps fed given normals (gibbs_sample_w_std :1011-1226) and LLW (:781-826)
    tau = np.linspace(3.0, 8.0, q)
    rm.set_tausq_inv(tau)
    z1, z2 = rng.standard_normal(n), rng.standard_normal(n)
    rm.deal_with_w(z1)
    out.update(tau=tau, z1=z1, z2=z2, w_sweep1=rm.w, llw_sweep1=rm.get_loglik_w(0)[0])
    rm.deal_with_w(z2)
    out.update(w_sweep2=rm.w, llw_sweep2=rm.get_loglik_w(0)[0])
    # ---- a proposal: BUILD of the other slot, accept, sweep again (theta_update :1420, accept_make_change :1432)
    th2 = pb["theta"] * (1 + .02 * rng.standard_normal(pb["theta"].size))
    rm.theta_update(1, th2)
    ok2, ll2, ld2 = rm.get_loglik_comps_w(1)
    assert ok2
    rm.accept_make_change()
    z3 = rng.standard_normal(n)
    rm.deal_with_w(z3)
    out.update(theta2=th2, loglik2=ll2, logdet2=ld2, z3=z3, w_sweep3=rm.w, llw_sweep3=rm.get_loglik_w(0)[0])
    rm.close()
    name = f"ref_q{q}_n{n}" + ("_limited" if limited else "") + ".npz"
    np.savez_compressed(os.path.join(HERE, name), **out)
    print(f"{name}: {len(out)} arrays, loglik {ll:.12g}")


# (q, n, limited, diag of mcmcsd, keep, burn, thin, adapting, sample_predicts): whole chains of the reference's OWN DRIVER,
# spamtree_mv_mcmc (spamtree_fit.cpp:5-430), on the host random stream shared with the oracle and the product (rng_mode 0)
CHAIN_CASES = [(2, 1200, False, 1e-7, 30, 40, 1, True, False), (3, 900, False, 1e-7, 24, 36, 2, True, True),
               (3, 1100, True, 1e-7, 20, 0, 1, False, False)]


def chain(q, n, limited, sd, keep, burn, thin, adapting, predicts, seed=31):
    from spamtree_b200 import synth
    pb = common.make_problem(q, n, limited=limited)
    d, t = pb["d"], pb["tree"]
    bounds, npar = synth.default_bounds(q), pb["theta"].size
    r = ref.spamtree_mv_mcmc(d["y"], d["X"], d["coords"], d["mv_id"], t["res_is_ref"], pb["csr"], limited, t["block_names"],
                             t["block_groups"], pb["beta"], pb["theta"], pb["tausq"], bounds, np.eye(npar) * sd, keep, burn, thin,
                             adapting=adapting, sample_predicts=predicts, seed=seed)
    th = r["theta_mcmc"]
    nmoves = int(np.sum(np.any(np.diff(th, axis=1) != 0, axis=0)))
    out = {"q": q, "n": n, "limited": int(limited), "blocking": t["blocking"], "sd": sd, "keep": keep, "burn": burn, "thin": thin,
           "adapting": int(adapting), "predicts": int(predicts), "seed": seed, "theta_mcmc": th, "beta_mcmc": r["beta_mcmc"],
           "tausq_mcmc": r["tausq_mcmc"], "paramsd": r["paramsd"], "w_saved": r["w_mcmc"][:, [0, keep // 2, keep - 1]],
           "yhat_saved": r["yhat_mcmc"][:, [0, keep // 2, keep - 1]], "block_ct_obs": r["block_ct_obs"],
           "parents_indexing_len": r["parents_indexing_len"]}
    name = f"ref_chain_q{q}_n{n}" + ("_limited" if limited else "") + ".npz"
    np.savez_compressed(os.path.join(HERE, name), **out)
    print(f"{name}: {keep} saved iterations, theta moved between {nmoves} of them")


if __name__ == "__main__":
    if not ref.available():
        raise SystemExit("oracle/_ref/libspamtree_ref.so is missing and the reference sources are not at " + ref.ref_src())
    which = sys.argv[1] if len(sys.argv) > 1 else "all"
    if which in ("all", "model"):
        for q, n, limited in CASES:
            one(q, n, limited)
    if which in ("all", "chain"):
        for c in CHAIN_CASES:
            chain(*c)
