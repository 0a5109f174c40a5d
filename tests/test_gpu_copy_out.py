"""Saved draws leave the device through one copy-out path (w_mcmc / yhat_mcmc of st_mcmc_run, the draws of st_predict_new)
and stay there through one draw store: host arrays the library cannot page-lock receive the same values as ordinary ones,
every combination of host arrays and device store gives the same arrays and summaries, and a run is not disturbed by the
run before it on the same handle."""
import ctypes as C
import itertools

import numpy as np
import pytest

import common
import spamtree_b200 as sb
from spamtree_b200 import _lib, synth

pytestmark = pytest.mark.gpu

SUMMARY_KEYS = ("mean", "sd", "quantiles", "mcse", "ess")


def _pinned(n):
    """n zeroed doubles of host memory that torch has page-locked already, so that the library's cudaHostRegister of the
    range is refused and its copies take the path for memory it could not page-lock"""
    import torch
    t = torch.zeros(n, dtype=torch.float64, pin_memory=True)
    rt = torch.cuda.cudart()
    err = rt.cudaHostRegister(t.data_ptr(), n * 8, 0)
    C.CDLL("libcudart.so.12").cudaGetLastError()  # (torch's runtime would report the refusal at its next launch check)
    if int(err) == 0:
        rt.cudaHostUnregister(t.data_ptr())
        pytest.fail("cudaHostRegister accepted host memory that torch had page-locked: the test would not reach the fallback")
    return t, t.numpy()


def _mcmc_into(gm, pb, keep, rng_mode, w, yh, seed=7, burn=2, thin=1):
    """st_mcmc_run with w_mcmc / yhat_mcmc pointing into the given arrays (None: not asked for)"""
    npar = pb["theta"].size
    b = np.ascontiguousarray(synth.default_bounds(pb["q"]).T, dtype=np.float64).reshape(-1)
    sd = np.ascontiguousarray(np.eye(npar) * 0.1)
    o = _lib.StMcmcOpts()
    o.set_unif_bounds, o.mcmcsd = b.ctypes.data_as(_lib.c_double_p), sd.ctypes.data_as(_lib.c_double_p)
    o.keep, o.burn, o.thin, o.adapting = keep, burn, thin, 1
    o.sample_beta = o.sample_tausq = o.sample_theta = o.sample_w = o.sample_predicts = 1
    o.faithful_beta_index, o.rng_mode, o.seed = 1, rng_mode, seed
    res = {"theta": np.zeros(npar * keep), "beta": np.zeros(gm.p * keep * gm.q), "tausq": np.zeros(gm.q * keep)}
    out = _lib.StMcmcOut()
    out.theta_mcmc, out.beta_mcmc, out.tausq_mcmc = [res[k].ctypes.data_as(_lib.c_double_p) for k in ("theta", "beta", "tausq")]
    out.w_mcmc = None if w is None else w.ctypes.data_as(_lib.c_double_p)
    out.yhat_mcmc = None if yh is None else yh.ctypes.data_as(_lib.c_double_p)
    gm._chk(_lib.lib.st_mcmc_run(gm._h, C.byref(o), C.byref(out)))
    res["n_accepted"] = out.n_accepted
    return res


@pytest.mark.parametrize("rng_mode,save_yhat", [(0, False), (0, True), (1, True)])
def test_arrays_that_cannot_be_page_locked(rng_mode, save_yhat):
    """rng_mode 0 saves w asynchronously only when yhat is not asked for (it forms yhat on the host from w)"""
    pb = common.make_problem(1, 625)
    keep = 6
    got, ref = {}, {}
    keep_alive = []
    for dst, pinned in ((got, True), (ref, False)):
        gm = common.product_model(pb, keep_H=False)
        for k in ("w", "yhat") if save_yhat else ("w",):
            if pinned:
                t, dst[k] = _pinned(gm.n_all * keep)
                keep_alive.append(t)
            else:
                dst[k] = np.zeros(gm.n_all * keep)
        dst["res"] = _mcmc_into(gm, pb, keep, rng_mode, dst["w"], dst.get("yhat"))
        gm.close()
    assert got["res"]["n_accepted"] == ref["res"]["n_accepted"]
    for k in ("theta", "beta", "tausq"):
        assert np.array_equal(got["res"][k], ref["res"][k]), k
    for k in ("w", "yhat") if save_yhat else ("w",):
        assert np.any(ref[k] != 0), k
        assert np.array_equal(got[k], ref[k]), k


def test_predict_new_into_arrays_that_cannot_be_page_locked():
    pb = common.make_problem(1, 625)
    d = pb["d"]
    miss = np.isnan(d["y"])
    cn, xn, mvn = d["coords"][miss], d["X"][miss], d["mv_id"][miss]
    tn = sb.make_tree(d["coords"], d["y"], d["mv_id"], cell_size=25, seed=0, coords_new=cn, mv_id_new=mvn)["new"]
    gm = common.product_model(pb, keep_H=False)
    res = gm.mcmc(synth.default_bounds(1), np.eye(4) * 0.1, 9, 3, 2, adapting=True, rng_mode=1, seed=7)
    nn, S = cn.shape[0], res["theta_mcmc"].shape[1]
    cm = np.ascontiguousarray(cn.T).reshape(-1)
    xm = np.ascontiguousarray(xn.T).reshape(-1)
    mv = np.ascontiguousarray(mvn, dtype=np.int64)
    grp, pp, pi = [np.ascontiguousarray(tn[k], dtype=np.int64) for k in ("group", "parents_ptr", "parents_idx")]
    r = _lib.StNewRows()
    r.n_new, r.coords, r.mv_id, r.X = nn, cm.ctypes.data_as(_lib.c_double_p), mv.ctypes.data_as(_lib.c_int64_p), xm.ctypes.data_as(_lib.c_double_p)
    r.n_groups = pp.size - 1
    r.group, r.parents_ptr, r.parents_idx = [a.ctypes.data_as(_lib.c_int64_p) for a in (grp, pp, pi)]
    th = np.ascontiguousarray(res["theta_mcmc"].T).reshape(-1)
    be = np.ascontiguousarray(res["beta_mcmc"].transpose(2, 1, 0)).reshape(-1)
    ta = np.ascontiguousarray(res["tausq_mcmc"].T).reshape(-1)
    w = np.ascontiguousarray(res["w_mcmc"])  # n_all x S, C order: one row's samples contiguous
    sm = _lib.StPredSamples()
    sm.n_samples = S
    sm.theta, sm.beta, sm.tausq, sm.w = [a.ctypes.data_as(_lib.c_double_p) for a in (th, be, ta, w)]
    sm.w_row_stride, sm.w_sample_stride, sm.seed = S, 1, 5
    outs = {}
    keep_alive = []
    for label, pinned in (("pinned", True), ("numpy", False)):
        a = {}
        for k in ("w_new", "y_new", "mean", "sd"):
            if pinned:
                t, a[k] = _pinned(nn * S)
                keep_alive.append(t)
            else:
                a[k] = np.zeros(nn * S)
        for k in ("w_mean", "w_sd", "y_mean", "y_sd"):
            a[k] = np.zeros(nn)
        o = _lib.StPredOut()
        for k, v in a.items():
            setattr(o, k, v.ctypes.data_as(_lib.c_double_p))
        gm._chk(_lib.lib.st_predict_new(gm._h, C.byref(r), C.byref(sm), C.byref(o)))
        outs[label] = a
    for k, v in outs["numpy"].items():
        assert np.any(v != 0), k
        assert np.array_equal(outs["pinned"][k], v), k
    gm.close()


MODES = ("none", "host", "store", "both")


def _run(pb, wmode, ymode, keep=7, seed=9):
    gm = common.product_model(pb, keep_H=False)
    ds = tuple(k for k, m in (("w", wmode), ("yhat", ymode)) if m in ("store", "both"))
    res = gm.mcmc(synth.default_bounds(pb["q"]), np.eye(pb["theta"].size) * 0.1, keep, 3, 2, adapting=True, rng_mode=1, seed=seed,
                  save_w=wmode in ("host", "both"), save_yhat=ymode in ("host", "both"), device_samples=ds)
    return gm, res


def test_every_combination_of_host_arrays_and_store():
    pb = common.make_problem(2, 1200)
    gref, ref = _run(pb, "host", "host")
    gboth, both = _run(pb, "both", "both")
    sref = {k: gboth.summarize(k, (0.1, 0.5, 0.9)) for k in ("w", "yhat")}
    gref.close()
    gboth.close()
    for k in ("w_mcmc", "yhat_mcmc", "theta_mcmc", "beta_mcmc", "tausq_mcmc", "paramsd"):
        assert np.array_equal(both[k], ref[k]), k
    for wmode, ymode in itertools.product(MODES, MODES):
        gm, res = _run(pb, wmode, ymode)
        for k in ("theta_mcmc", "beta_mcmc", "tausq_mcmc", "paramsd"):
            assert np.array_equal(res[k], ref[k]), (wmode, ymode, k)
        for q, key, mode in (("w", "w_mcmc", wmode), ("yhat", "yhat_mcmc", ymode)):
            if mode in ("host", "both"):
                assert np.array_equal(res[key], ref[key]), (wmode, ymode, key)
            else:
                assert res[key] is None
            if mode in ("store", "both"):
                s = gm.summarize(q, (0.1, 0.5, 0.9))
                for c in SUMMARY_KEYS:
                    assert np.array_equal(s[c], sref[q][c], equal_nan=True), (wmode, ymode, q, c)
            else:
                with pytest.raises(sb.SpamTreeError) as ex:
                    gm.summarize(q)
                assert ex.value.code == 1
        gm.close()


def test_second_run_with_different_keep():
    """the second run saves different quantities, with a different keep, from what the first run left on the handle"""
    pb = common.make_problem(1, 625)
    runs = (dict(keep=9, save_w=True, save_yhat=True, device_samples=("w", "yhat")),
            dict(keep=4, save_w=True, save_yhat=False, device_samples=("yhat",)),
            dict(keep=11, save_w=False, save_yhat=True, device_samples=()))
    twin_runs = [dict(r, save_w=True, save_yhat=True, device_samples=("w", "yhat")) for r in runs]
    gm, twin = common.product_model(pb, keep_H=False), common.product_model(pb, keep_H=False)
    for seed, (r, t) in enumerate(zip(runs, twin_runs)):
        kw = dict(adapting=True, rng_mode=1, seed=seed)
        bounds, sd = synth.default_bounds(1), np.eye(4) * 0.1
        a = gm.mcmc(bounds, sd, r["keep"], 2, 1, save_w=r["save_w"], save_yhat=r["save_yhat"], device_samples=r["device_samples"], **kw)
        b = twin.mcmc(bounds, sd, t["keep"], 2, 1, save_w=True, save_yhat=True, device_samples=("w", "yhat"), **kw)
        for k in ("theta_mcmc", "beta_mcmc", "tausq_mcmc", "paramsd"):
            assert np.array_equal(a[k], b[k]), (seed, k)
        for q, key in (("w", "w_mcmc"), ("yhat", "yhat_mcmc")):
            if r["save_" + q]:
                assert np.array_equal(a[key], b[key]), (seed, key)
            if q in r["device_samples"]:
                sa, sb_ = gm.summarize(q), twin.summarize(q)
                assert all(np.array_equal(sa[c], sb_[c], equal_nan=True) for c in SUMMARY_KEYS), (seed, q)
            else:
                with pytest.raises(sb.SpamTreeError):
                    gm.summarize(q)
    gm.close()
    twin.close()
