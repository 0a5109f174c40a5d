"""The kernels under every launch plan the planner can choose, against the CPU oracle at 1e-9.

test_gpu_parity.py runs the planner's default choices on make_tree() problems, which at its sizes leave most of the plan's
branches alone: work groups of one or two blocks, no parent with more than a few children, no block above 49 rows.  Here
the same checks run under each configuration of the plan (environment variables read at handle creation, or
smem_panel_bytes) and on hand-built trees (shape_trees.py) whose shapes reach the other branches: multi-block work groups
and paired warps, single and double cp.async rings, 4/8/16-warp CTAs, the untabulated Gram lookups (more than 64 children,
more than 256 (child, tile) pairs), several Gram item rounds and row chunks, register and general factorisations at
m = 32 / 33, leaves of a full work group, chains 32 deep, all-NaN siblings.  test_plan_envelope.py checks on the CPU that
each configuration reaches its path.

Per (problem, configuration), on a keep_H = True handle: the log-density of both slots, H and Ri of every observed block,
the per-block log-density pieces, w after two sweeps with shared z and one without noise, the Sigi_tot / Smu_tot probes of
every block, LLW, predict, a proposal that is accepted, the swap and one more sweep.  A keep_H = False handle (the
deferred childless level, what spamtree() and the benchmark run) of the same configuration must give the same w (bit for
bit where its BUILD launches are the same).  Configurations that only change scheduling or buffering must give their
baseline's numbers bit for bit (see below)."""
import numpy as np
import pytest

import common
import launch_configs as lc
from common import relerr
from dense_twin import block_truth_ld
from spamtree_b200 import synth

pytestmark = pytest.mark.gpu
TOL = 1e-9

# Bit-identical to the baseline, from the code: ST_BUILD_NS changes how many stages of the chain factor's rows are in
# flight (st_build.cu: the ring), not which products are summed in which order; ST_GRAM_ROOM changes how many rows
# gram_level_kernel stages per chunk, while every thread still adds the rows in order into the same registers; ST_PDL,
# ST_OVERLAP and ST_LLW_OVERLAP only change when kernels start (programmatic dependent launch, second streams); ST_DEFER=0
# gives a keep_H = False handle the plan of a keep_H = True one.  The others change which sibling blocks share a work
# group and so the CTA width and the paired-warp split of the reductions (npair): held to the oracle tolerance only.
# launch_configs.py lists the rows; test_plan_envelope.py checks that each reaches its path.
CONFIGS, ROWS = lc.CONFIGS, lc.ROWS
_ids = [f"{p}-{c}" for p, c in ROWS]

_cache = {}


def _script(m, pb, full):
    """the sequence every model runs; full: also the per-block state (keep_H handles and the oracle)"""
    rng = np.random.default_rng(11)
    n, nb = pb["n"], pb["tree"]["n_blocks"]
    th2 = pb["theta"] * (1 + 2e-3 * rng.standard_normal(pb["theta"].size))
    y = pb["d"]["y"]
    ip, ii = pb["tree"]["indexing_ptr"], pb["tree"]["indexing_idx"]
    obs = np.array([np.isfinite(y[ii[ip[u]:ip[u + 1]]]).any() for u in range(nb)])
    npar = np.diff(pb["tree"]["parents_ptr"])
    r = {}
    m.w = rng.standard_normal(n) * .5
    r["build0"], r["build1"] = m.get_loglik_comps_w(0), m.get_loglik_comps_w(1)
    if full:
        r["H"] = {u: m.get("H", u) if hasattr(m, "get") else m.node_state("H", u) for u in range(nb) if obs[u] and npar[u]}
        r["Ri"] = {u: _ri(m, u) for u in range(nb) if obs[u]}
        for k in ("logdetCi_comps", "loglik_w_comps"):
            r[k] = m.get(k) if hasattr(m, "get") else m.node_state(k)
    zs = [rng.standard_normal(n), rng.standard_normal(n), np.zeros(n)]
    for i, z in enumerate(zs):
        m.deal_with_w(z)
        r[f"w{i}"] = m.w
    if full:
        for k in ("Sigi_tot", "Smu_tot"):
            r[k] = {u: m.get(k, u) if hasattr(m, "get") else m.node_state(k, u) for u in range(nb) if obs[u]}
    r["llw"] = m.get_loglik_w(0)
    m.predict(True)
    r["w_pred"] = m.w
    m.theta_update(1, th2)
    r["proposal"] = m.get_loglik_comps_w(1)
    m.accept_make_change()
    r["llw_swapped"] = m.get_loglik_w(0)
    m.deal_with_w(rng.standard_normal(n))
    r["w_swapped"] = m.w
    r["llw_end"] = m.get_loglik_w(0)
    return r


def _ri(m, u):
    if hasattr(m, "get"):  # oracle
        return m.get("Ri", u) if m.geti("block_is_reference")[u] else m.get("ccholprecdiag", u)
    return m.node_state("Ri", u)


def _oracle(name):
    """the oracle's run of the script, and the bound for the per-block state: 1e-9, or where the oracle's own rounding is
    larger (deep chains: it forms K_pa^-1 explicitly), 4 x its distance from the extended-precision truth on the blocks with
    the largest parent sets (test_gpu_fullsize.py does the same at full size)"""
    if ("oracle", name) in _cache:
        return _cache[("oracle", name)]
    pb = lc.problem(name)
    om = common.oracle_model(pb)
    r = _script(om, pb, True)
    isref = om.geti("block_is_reference")
    om.close()
    t = pb["tree"]
    ip, ii, pp, pi = t["indexing_ptr"], t["indexing_idx"], t["parents_ptr"], t["parents_idx"]
    deep = sorted(r["H"], key=lambda u: -(pp[u + 1] - pp[u]) * 10**6 - sum(ip[a + 1] - ip[a] for a in pi[pp[u]:pp[u + 1]]))[:3]
    worst = 0.0
    truth = {}
    for u in deep:
        ru = ii[ip[u]:ip[u + 1]]
        rp = np.concatenate([ii[ip[a]:ip[a + 1]] for a in pi[pp[u]:pp[u + 1]]])
        Ht, Rt = block_truth_ld(pb["d"]["coords"], pb["d"]["mv_id"], ru, rp, pb["theta"], pb["q"], bool(isref[u]))
        m = ru.size
        Ho = r["H"][u].reshape(-1, m).T
        Ro = r["Ri"][u].reshape(m, m).T if isref[u] else r["Ri"][u]
        worst = max(worst, _ldrel(Ho, Ht), _ldrel(Ro, Rt))
        truth[u] = (Ht, Rt, bool(isref[u]))
    out = (r, max(TOL, 4 * worst), truth)
    _cache[("oracle", name)] = out
    return out


def _ldrel(a, b):
    return float(np.max(np.abs(a.astype(np.longdouble) - b)) / np.max(np.abs(b)))


def _run(name, config, keep_H, monkeypatch):
    key = ("run", name, config, keep_H)
    if key in _cache:
        return _cache[key]
    c = CONFIGS[config]
    with monkeypatch.context() as mp:
        for k, v in c["env"].items():
            mp.setenv(k, v)
        pb = lc.problem(name)
        gm = common.product_model(pb, keep_H=keep_H, **c["kw"])
    try:
        r = _script(gm, pb, keep_H)
    finally:
        gm.close()
    _cache[key] = r
    return r


def _rel(a, b):
    return abs(a - b) / abs(b)


@pytest.mark.parametrize("name,config", ROWS, ids=_ids)
def test_launch_plan_matches_oracle(name, config, monkeypatch):
    ro, slack, truth = _oracle(name)
    rg = _run(name, config, True, monkeypatch)
    for k in ("build0", "build1", "proposal"):
        assert rg[k][0] and ro[k][0], k
        assert _rel(rg[k][1], ro[k][1]) <= TOL and _rel(rg[k][2], ro[k][2]) <= TOL, (k, rg[k], ro[k])
    for k in ("llw", "llw_swapped", "llw_end"):
        assert _rel(rg[k][0], ro[k][0]) <= TOL, (k, rg[k], ro[k])
    err = {k: max((relerr(rg[k][u], ro[k][u]) for u in ro[k]), default=0.0) for k in ("H", "Ri", "Sigi_tot", "Smu_tot")}
    err.update({k: relerr(rg[k], ro[k]) for k in ("logdetCi_comps", "loglik_w_comps", "w0", "w1", "w2", "w_pred", "w_swapped")})
    # the per-block log-density pieces of a w that is not a draw from the model get one more digit (as at full size)
    bad = {k: v for k, v in err.items() if not v <= (10 * slack if k == "loglik_w_comps" else slack)}
    assert not bad, (bad, slack)
    pb = lc.problem(name)
    ip = pb["tree"]["indexing_ptr"]
    for u, (Ht, Rt, isref) in truth.items():  # the GPU against the truth where the oracle is least accurate
        m = ip[u + 1] - ip[u]
        Ri = rg["Ri"][u].reshape(m, m).T if isref else rg["Ri"][u]
        assert _ldrel(rg["H"][u].reshape(-1, m).T, Ht) <= TOL and _ldrel(Ri, Rt) <= TOL, u


@pytest.mark.parametrize("name,config", ROWS, ids=_ids)
def test_deferred_handle_equals_eager_handle(name, config, monkeypatch):
    """keep_H = False defers the backward half of BUILD at the childless level to the swap.  The deferred panel carries one
    more column (w_pa), which can change how the level's blocks are grouped and which column tiles get paired warps
    (16-row leaves: 2 tiles and 2 paired warps become 3 tiles and 1), and so the order of the reductions.  Where the two
    handles' BUILD work groups are the same (blocks, columns, CTA width, paired warps), w is the same bit for bit;
    otherwise it agrees to rounding.  The deferred forward half sums the childless level's log-density from Z, in another
    order: 1e-12 unless no level is deferred."""
    re = _run(name, config, True, monkeypatch)
    rd = _run(name, config, False, monkeypatch)
    same_launches = np.array_equal(lc.plan(name, config, keep_H=True, which="build_groups"),
                                   lc.plan(name, config, keep_H=False, which="build_groups"))
    deferred = any(v["deferrable"] for v in lc.plan(name, config, keep_H=False)[1])
    for k in ("w0", "w1", "w2", "w_pred", "w_swapped"):
        if same_launches:
            assert np.array_equal(rd[k], re[k]), k
        else:
            assert relerr(rd[k], re[k]) <= 1e-12, (k, relerr(rd[k], re[k]))
    dtol = 1e-12 if deferred else 0.0
    for k in ("build0", "build1", "proposal"):  # (acceptable, loglik, logdet)
        assert re[k][0] == rd[k][0]
        assert all(_rel(a, b) <= dtol for a, b in zip(re[k][1:], rd[k][1:])), (k, re[k], rd[k])
    for k in ("llw", "llw_swapped", "llw_end"):
        assert all(_rel(a, b) <= dtol for a, b in zip(re[k], rd[k])), (k, re[k], rd[k])


BITWISE = [(p, c) for p, c in ROWS if c != "default" and CONFIGS[c]["bitwise"]]


@pytest.mark.parametrize("name,config", BITWISE, ids=[f"{p}-{c}" for p, c in BITWISE])
def test_scheduling_configurations_are_bit_identical(name, config, monkeypatch):
    base = CONFIGS[config]["base"]
    # (ST_DEFER=0: the keep_H = False handle against the keep_H = True handle of the baseline, whose plan it takes)
    pairs = [(False, True)] if config == "defer0" else [(True, True), (False, False)]
    for kc, kb in pairs:
        rd, rc = _run(name, base, kb, monkeypatch), _run(name, config, kc, monkeypatch)
        for k, v in rc.items():
            if isinstance(v, dict):
                assert all(np.array_equal(v[u], rd[k][u]) for u in v), (kc, k)
            elif isinstance(v, tuple):
                assert v == rd[k], (kc, k, v, rd[k])
            else:
                assert np.array_equal(v, rd[k]), (kc, k)


@pytest.mark.parametrize("config", lc.CHAIN_CONFIGS)
def test_device_resident_chain_under_configuration(config, monkeypatch):
    """a short device-resident chain (rng_mode 1, the benchmark's handle: keep_H = False) under the configuration.  Where
    the configuration only changes scheduling and its BUILD work groups are the default's, the chain must be the default's
    bit for bit.  Otherwise (ST_SPREAD=0: other work groups and reduction orders) it must match the host replay of
    test_gpu_device_chain.py run under the same configuration, as test_device_chain_equals_host_replay requires of the
    default."""
    from test_gpu_device_chain import _replay
    pb = lc.problem(lc.CHAIN_PROBLEM)
    bounds, sd0 = synth.default_bounds(3), np.eye(pb["theta"].size) * 1e-4
    keep, burn, thin, seed = 10, 4, 1, 31
    env = CONFIGS[config]["env"]

    def chain(env):
        with monkeypatch.context() as mp:
            for k, v in env.items():
                mp.setenv(k, v)
            gm = common.product_model(pb, keep_H=False)
        try:
            return gm.mcmc(bounds, sd0, keep, burn, thin, adapting=True, faithful_beta_index=True, rng_mode=1, seed=seed)
        finally:
            gm.close()

    rc = chain(env)
    assert rc["n_accepted"] > 0
    same_launches = np.array_equal(lc.plan(lc.CHAIN_PROBLEM, config, which="build_groups"),
                                   lc.plan(lc.CHAIN_PROBLEM, "default", keep_H=False, which="build_groups"))
    if CONFIGS[config]["bitwise"] and same_launches:
        if ("chain", "default") not in _cache:
            _cache[("chain", "default")] = chain({})
        rd = _cache[("chain", "default")]
        assert rd["n_accepted"] == rc["n_accepted"]
        for k in ("theta_mcmc", "beta_mcmc", "tausq_mcmc", "w_mcmc", "yhat_mcmc", "paramsd"):
            assert np.array_equal(rd[k], rc[k]), k
        return
    with monkeypatch.context() as mp:
        for k, v in env.items():
            mp.setenv(k, v)
        h = _replay(pb, bounds, sd0, keep, burn, thin, seed, True)
    assert rc["n_accepted"] == h["acc"]
    err = {"theta": relerr(rc["theta_mcmc"], np.array(h["theta"]).T), "beta": relerr(rc["beta_mcmc"], np.array(h["beta"]).transpose(1, 0, 2)),
           "tausq": relerr(rc["tausq_mcmc"], np.array(h["tausq"]).T), "paramsd": relerr(rc["paramsd"], h["paramsd"]),
           "w": relerr(rc["w_mcmc"], np.array(h["w"]).T), "yhat": relerr(rc["yhat_mcmc"], np.array(h["yhat"]).T)}
    assert all(v <= TOL for v in err.values()), err
