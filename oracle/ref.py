"""ctypes wrapper of oracle/_ref/libspamtree_ref.so — the reference's OWN model layer (spamtree_model.cpp,
covariance_functions.cpp, tree_utils.cpp, tree_dep.cpp, mh_adapt.cpp), compiled unmodified from the reference package's
src/ directory against the Armadillo/Rcpp stand-in in oracle/refshim/.  TEST INFRASTRUCTURE ONLY: it pins the CPU oracle.
The library is built by `make -C oracle ref` wherever that directory exists (ref_src())."""
import ctypes as C
import json
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_ref", "libspamtree_ref.so")
_dp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_int64)
_lib = None


def ref_src():
    """the reference package's src/ directory: SPAMTREE_REF_SRC if set, else src/ under BASELINE.json's reference_path"""
    src = os.environ.get("SPAMTREE_REF_SRC")
    if not src:
        with open(os.path.join(os.path.dirname(_HERE), "BASELINE.json")) as f:
            src = os.path.join(json.load(f)["reference_path"], "src")
    return src


def build(stdout=subprocess.DEVNULL, stderr=None):
    subprocess.check_call(["make", "-C", _HERE, "ref", "REFSRC=" + ref_src()], stdout=stdout, stderr=stderr)


def available():
    if not os.path.exists(LIB_PATH) and os.path.isdir(ref_src()):
        try:
            build(stderr=subprocess.DEVNULL)
        except Exception:
            return False
    return os.path.exists(LIB_PATH)


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(LIB_PATH)
        L.ref_create.restype = C.c_void_p
        L.ref_create.argtypes = [C.c_int64, C.c_int, C.c_int, _dp, _dp, _dp, _ip, C.c_int, _ip, _ip, _ip, _ip, _ip, _ip, _dp, _dp, _ip,
                                 C.c_int, C.c_int, _dp, C.c_int, _dp, C.c_double]
        L.ref_destroy.argtypes = [C.c_void_p]
        L.ref_seed.argtypes = [C.c_void_p, C.c_uint64]
        L.ref_theta_update.argtypes = [C.c_void_p, C.c_int, _dp]
        L.ref_build.restype = C.c_int
        L.ref_build.argtypes = [C.c_void_p, C.c_int, _dp]
        L.ref_loglik_w.argtypes = [C.c_void_p, C.c_int, _dp]
        L.ref_gibbs.restype = C.c_int
        L.ref_gibbs.argtypes = [C.c_void_p, _dp]
        L.ref_swap.argtypes = [C.c_void_p]
        L.ref_predict.argtypes = [C.c_void_p, C.c_int]
        L.ref_sample_beta.argtypes = [C.c_void_p, _dp]
        L.ref_sample_tausq.argtypes = [C.c_void_p, _dp]
        L.ref_get_w.argtypes = [C.c_void_p, _dp]
        L.ref_set_w.argtypes = [C.c_void_p, _dp]
        L.ref_set_tausq_inv.argtypes = [C.c_void_p, _dp]
        L.ref_get_params.argtypes = [C.c_void_p, _dp, _dp, _dp]
        L.ref_get.restype = C.c_int64
        L.ref_get.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int, _dp, C.c_int64]
        L.ref_kthresholds.argtypes = [_dp, C.c_int64, C.c_int, _dp]
        L.ref_cross_covariance_ag10.argtypes = [_dp, _ip, C.c_int64, _dp, _ip, C.c_int64, _dp, _dp, _dp, _dp, C.c_int, _dp, C.c_int, _dp]
        L.ref_number_revalue.argtypes = [_ip, C.c_int64, C.c_int, _ip, _ip, C.c_int64, _ip]
        L.ref_make_edges.restype = C.c_int
        L.ref_make_edges.argtypes = [_dp, C.c_int64, C.c_int, _ip, C.c_int64, _ip, C.c_int, _ip, _ip, _ip, _ip, _ip]
        L.ref_part_axis_parallel_lmt.argtypes = [_dp, C.c_int64, C.c_int, _dp, _ip, _dp]
        L.ref_ram_adapt.restype = C.c_int
        L.ref_ram_adapt.argtypes = [C.c_int, _dp, C.c_int, _dp, _dp, _dp, _dp]
        L.ref_propose.argtypes = [C.c_int, _dp, _dp, _dp, _dp, _dp]
        L.ref_do_i_accept.restype = C.c_int
        L.ref_do_i_accept.argtypes = [C.c_double, C.c_double]
        L.ref_spamtree_mv_mcmc.restype = C.c_int
        L.ref_spamtree_mv_mcmc.argtypes = [C.c_int64, C.c_int, C.c_int, _dp, _dp, _dp, _ip, C.c_int, _ip, _ip, _ip, _ip, _ip, _ip, _dp, _dp,
                                           _ip, C.c_int, C.c_int, _dp, C.c_int, _dp, C.c_double, _dp, _dp, C.c_int, C.c_int, C.c_int,
                                           C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, _dp, _dp, _dp, _dp, _dp,
                                           _dp, _ip, _ip]
        _lib = L
    return _lib


def _f(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _i(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _pd(a):
    return None if a is None else a.ctypes.data_as(_dp)


def _pi(a):
    return None if a is None else a.ctypes.data_as(_ip)


def _cm(a):
    a = np.asarray(a, dtype=np.float64)
    return _f(a.T).reshape(-1) if a.ndim == 2 else _f(a).reshape(-1)


class RefModel:
    """the reference's SpamTreeMV (src/spamtree_model.h:22-212), same call surface as oracle.OracleModel"""

    def __init__(self, y, X, coords, mv_id, res_is_ref, csr, limited_tree, block_names, block_groups, beta, theta, tausq):
        L = lib()
        self.y = _f(y).reshape(-1)
        self.n_all = self.y.size
        Xa = np.asarray(X, dtype=np.float64).reshape(self.n_all, -1)
        self.p, self.mv = Xa.shape[1], _i(mv_id)
        self.q = int(np.unique(self.mv).size)
        self._keep = [_cm(Xa), _cm(coords)] + [_i(a) for a in csr] + [_f(block_names), _f(block_groups), _i(res_is_ref), _f(theta), _f(beta)]
        Xc, cc, ip, ii, pp, pi, cp, ci, bn, bg, rr, th, be = self._keep
        self.n_blocks = ip.size - 1
        self.h = L.ref_create(self.n_all, self.p, self.q, _pd(self.y), _pd(Xc), _pd(cc), _pi(self.mv), self.n_blocks, _pi(ip), _pi(ii),
                              _pi(pp), _pi(pi), _pi(cp), _pi(ci), _pd(bn), _pd(bg), _pi(rr), rr.size, int(bool(limited_tree)), _pd(th),
                              th.size, _pd(be), float(tausq))
        if not self.h:
            raise RuntimeError("reference model construction failed")

    def close(self):
        if getattr(self, "h", None):
            lib().ref_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def seed(self, s):
        lib().ref_seed(self.h, int(s))

    def theta_update(self, slot, theta):
        t = _f(theta)
        lib().ref_theta_update(self.h, slot, _pd(t))

    def get_loglik_comps_w(self, slot):
        o = np.zeros(3)
        ok = lib().ref_build(self.h, slot, _pd(o))
        return bool(ok), float(o[0]), float(o[1])

    def get_loglik_w(self, slot=0):
        o = np.zeros(2)
        lib().ref_loglik_w(self.h, slot, _pd(o))
        return float(o[0]), float(o[1])

    def deal_with_w(self, z=None):
        zz = None if z is None else _f(z)
        if not lib().ref_gibbs(self.h, _pd(zz)):
            raise RuntimeError("Error at gibbs_sample_w")

    def accept_make_change(self):
        lib().ref_swap(self.h)

    def predict(self, theta_changed=True):
        lib().ref_predict(self.h, int(bool(theta_changed)))

    def gibbs_sample_beta(self, zb=None):
        z = None if zb is None else _cm(zb)
        lib().ref_sample_beta(self.h, _pd(z))

    def gibbs_sample_tausq(self, fixed=None):
        f = None if fixed is None else _f(fixed)
        lib().ref_sample_tausq(self.h, _pd(f))

    @property
    def w(self):
        o = np.zeros(self.n_all)
        lib().ref_get_w(self.h, _pd(o))
        return o

    @w.setter
    def w(self, v):
        a = _f(v)
        lib().ref_set_w(self.h, _pd(a))

    def set_tausq_inv(self, t):
        a = _f(t)
        lib().ref_set_tausq_inv(self.h, _pd(a))

    def params(self):
        B, t, xb = np.zeros(self.p * self.q), np.zeros(self.q), np.zeros(self.n_all)
        lib().ref_get_params(self.h, _pd(B), _pd(t), _pd(xb))
        return {"Bcoeff": B.reshape(self.q, self.p).T.copy(), "tausq_inv": t, "XB": xb}

    def get(self, name, u=0, slot=0, c=0):
        n = lib().ref_get(self.h, name.encode(), slot, int(u), int(c), None, 0)
        if n < 0:
            raise KeyError(name)
        o = np.zeros(max(n, 1))
        lib().ref_get(self.h, name.encode(), slot, int(u), int(c), _pd(o), o.size)
        return o[:n]

    def geti(self, name, u=0, slot=0, c=0):
        return self.get(name, u, slot, c).astype(np.int64)


def kthresholds(x, k):
    x = _f(x)
    res = np.zeros(max(k - 1, 0))
    lib().ref_kthresholds(_pd(x), x.size, k, _pd(res))
    return res


def cross_covariance_ag10(coords1, mv1, coords2, mv2, ai1, ai2, phi_i, thetamv, Dmat):
    c1, c2 = np.asarray(coords1, dtype=np.float64), np.asarray(coords2, dtype=np.float64)
    n1, n2 = c1.shape[0], c2.shape[0]
    Dm = np.asarray(Dmat, dtype=np.float64)
    q = Dm.shape[1]
    a, b, m1, m2 = _cm(c1), _cm(c2), _i(mv1), _i(mv2)
    A1, A2, PH, TM, DD = _f(ai1), _f(ai2), _f(phi_i), _f(np.atleast_1d(thetamv)), _cm(Dm)
    out = np.zeros(n1 * n2)
    lib().ref_cross_covariance_ag10(_pd(a), _pi(m1), n1, _pd(b), _pi(m2), n2, _pd(A1), _pd(A2), _pd(PH), _pd(TM), TM.size, _pd(DD), q, _pd(out))
    return out.reshape(n2, n1).T.copy()


def number_revalue(original_mat, from_val, to_val):
    om = np.asarray(original_mat, dtype=np.int64)
    nr, nc = om.shape
    flat, fv, tv = _i(om.T.reshape(-1)), _i(from_val), _i(to_val)
    out = np.zeros(nr * nc, dtype=np.int64)
    lib().ref_number_revalue(_pi(flat), nr, nc, _pi(fv), _pi(tv), fv.size, _pi(out))
    return out.reshape(nc, nr).T.copy()


def make_edges(parchimat, non_empty_blocks, res_is_ref, limited=False):
    """the reference's make_edges / make_edges_limited (tree_dep.cpp:75-186): lists of 0-based ids per block"""
    pm = np.asarray(parchimat, dtype=np.float64)
    nr, L = pm.shape
    flat, ne, rr = _cm(pm), _i(non_empty_blocks), _i(res_is_ref)
    counts = np.zeros(3, dtype=np.int64)
    if lib().ref_make_edges(_pd(flat), nr, L, _pi(ne), ne.size, _pi(rr), int(limited), None, None, None, None, _pi(counts)):
        raise RuntimeError("reference make_edges threw")
    nb = int(counts[0])
    pp, pi = np.zeros(nb + 1, np.int64), np.zeros(max(int(counts[1]), 1), np.int64)
    cp, ci = np.zeros(nb + 1, np.int64), np.zeros(max(int(counts[2]), 1), np.int64)
    lib().ref_make_edges(_pd(flat), nr, L, _pi(ne), ne.size, _pi(rr), int(limited), _pi(pp), _pi(pi), _pi(cp), _pi(ci), _pi(counts))
    return {"parents": [pi[pp[i]:pp[i + 1]].copy() for i in range(nb)], "children": [ci[cp[i]:cp[i + 1]].copy() for i in range(nb)]}


def part_axis_parallel_lmt(coords, thresholds):
    """tree_dep.cpp:58-67"""
    coords = np.asarray(coords, dtype=np.float64)
    n, d = coords.shape
    ptr = np.zeros(d + 1, dtype=np.int64)
    for j in range(d):
        ptr[j + 1] = ptr[j] + len(thresholds[j])
    thr = _f(np.concatenate([np.asarray(t, dtype=np.float64) for t in thresholds]) if ptr[-1] else np.zeros(1))
    cm, out = _cm(coords), np.zeros(n * d)
    lib().ref_part_axis_parallel_lmt(_pd(cm), n, d, _pd(thr), _pi(ptr), _pd(out))
    return out.reshape(d, n).T.copy()


def ram_adapt(metropolis_sd, U, alpha):
    """the reference's RAMAdapt (mh_adapt.h:40-135) over a recorded sequence: U (steps x npar), alpha (steps);
    returns (final paramsd, trace steps x npar x npar)"""
    U = np.asarray(U, dtype=np.float64)
    steps, npar = U.shape
    sd, uu, al = _cm(metropolis_sd), _f(U.reshape(-1)), _f(alpha)
    out, tr = np.zeros(npar * npar), np.zeros(steps * npar * npar)
    if lib().ref_ram_adapt(npar, _pd(sd), steps, _pd(uu), _pd(al), _pd(out), _pd(tr)):
        raise RuntimeError("reference RAMAdapt threw (chol failed)")
    return out.reshape(npar, npar).T.copy(), tr.reshape(steps, npar, npar).transpose(0, 2, 1).copy()


def propose(param, bounds, paramsd, U):
    """spamtree_fit.cpp:211-215 + calc_jacobian (mh_adapt.h:230-239): (new_param, jacobian, out_of_bounds)"""
    par, B, sd, u = _f(param), _cm(bounds), _cm(paramsd), _f(U)
    out = np.zeros(par.size + 2)
    lib().ref_propose(par.size, _pd(par), _pd(B), _pd(sd), _pd(u), _pd(out))
    return out[:par.size].copy(), float(out[par.size]), bool(out[par.size + 1])


def do_i_accept(logaccept, u):
    return bool(lib().ref_do_i_accept(float(logaccept), float(u)))


def spamtree_mv_mcmc(y, X, coords, mv_id, res_is_ref, csr, limited_tree, block_names, block_groups, beta, theta, tausq, bounds, mcmcsd,
                     keep, burn, thin, adapting=True, sample_beta=True, sample_tausq=True, sample_theta=True, sample_w=True,
                     sample_predicts=True, seed=1):
    """the reference's OWN driver spamtree_mv_mcmc (spamtree_fit.cpp:5-430), its R-side random numbers replaced by the host
    stream the oracle and the product use (seeded with `seed`)"""
    y = _f(y).reshape(-1)
    n = y.size
    Xa = np.asarray(X, dtype=np.float64).reshape(n, -1)
    p, mv = Xa.shape[1], _i(mv_id)
    q = int(np.unique(mv).size)
    Xc, cc = _cm(Xa), _cm(coords)
    ip, ii, pp, pi, cp, ci = [_i(a) for a in csr]
    bn, bg, rr, th, be = _f(block_names), _f(block_groups), _i(res_is_ref), _f(theta), _f(beta)
    nb, npar = ip.size - 1, th.size
    B, sd = _cm(bounds), _cm(mcmcsd)
    bm, tm, thm = np.zeros(p * keep * q), np.zeros(q * keep), np.zeros(npar * keep)
    w, yh, psd = np.zeros(n * keep), np.zeros(n * keep), np.zeros(npar * npar)
    bco, pil = np.zeros(nb, dtype=np.int64), np.zeros(nb, dtype=np.int64)
    rc = lib().ref_spamtree_mv_mcmc(n, p, q, _pd(y), _pd(Xc), _pd(cc), _pi(mv), nb, _pi(ip), _pi(ii), _pi(pp), _pi(pi), _pi(cp), _pi(ci),
                                    _pd(bn), _pd(bg), _pi(rr), rr.size, int(bool(limited_tree)), _pd(th), npar, _pd(be), float(tausq),
                                    _pd(B), _pd(sd), keep, burn, thin, int(adapting), int(sample_beta), int(sample_tausq),
                                    int(sample_theta), int(sample_w), int(sample_predicts), int(seed), _pd(bm), _pd(tm), _pd(thm), _pd(w),
                                    _pd(yh), _pd(psd), _pi(bco), _pi(pil))
    if rc:
        raise RuntimeError("the reference's spamtree_mv_mcmc threw")
    return {"w_mcmc": w.reshape(keep, n).T.copy(), "yhat_mcmc": yh.reshape(keep, n).T.copy(),
            "beta_mcmc": bm.reshape(q, keep, p).transpose(2, 1, 0).copy(), "tausq_mcmc": tm.reshape(keep, q).T.copy(),
            "theta_mcmc": thm.reshape(keep, npar).T.copy(), "paramsd": psd.reshape(npar, npar).T.copy(),
            "block_ct_obs": bco, "parents_indexing_len": pil}
