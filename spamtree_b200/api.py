"""Host-side mirror of the reference's public interface for the hot path.

R is not available in this environment, so the R-level entry point `spamtree()` (R/spamtree_fit.R:1-371) and the Rcpp
export `spamtree_mv_mcmc` (src/spamtree_fit.cpp:5-54) are mirrored here in Python with the same argument names,
defaults and return keys; the model layer `SpamTreeMV` (src/spamtree_model.h:22-212) is a thin wrapper over the C ABI.
All compute happens in libspamtree_b200.so (CUDA, sm_100a); nothing here falls back to the CPU.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import lib

_ERRORS = {1: "invalid argument", 2: "CUDA error", 3: "not positive definite", 4: "unsupported", 5: "NaN log-likelihood"}


class SpamTreeError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[{_ERRORS.get(code, code)}] {msg}")
        self.code = code


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _dp(a):
    return None if a is None else a.ctypes.data_as(_lib.c_double_p)


def _ip(a):
    return None if a is None else a.ctypes.data_as(_lib.c_int64_p)


def _colmajor(a):
    """column-major (Fortran) flattening, as arma::mat memory"""
    return _f64(np.asarray(a, dtype=np.float64).T).reshape(-1) if np.ndim(a) == 2 else _f64(a).reshape(-1)


def lists_to_csr(lists):
    ptr = np.zeros(len(lists) + 1, dtype=np.int64)
    for i, l in enumerate(lists):
        ptr[i + 1] = ptr[i] + len(l)
    idx = np.concatenate([np.asarray(l, dtype=np.int64) for l in lists]) if len(lists) and ptr[-1] > 0 else np.zeros(0, np.int64)
    return ptr, _i64(idx)


def csr_to_lists(ptr, idx):
    return [np.asarray(idx[ptr[i]:ptr[i + 1]], dtype=np.int64) for i in range(len(ptr) - 1)]


# --------------------------------------------------------------------------------------------- tree_dep.cpp exports
def kthresholds(x, k):
    """tree_dep.cpp:16-27"""
    x = _f64(x)
    res = np.zeros(max(k - 1, 0))
    rc = lib.st_kthresholds(_dp(x), x.size, int(k), _dp(res))
    if rc:
        raise SpamTreeError(rc, "st_kthresholds")
    return res


def part_axis_parallel_lmt(coords, thresholds):
    """tree_dep.cpp:58-67; thresholds: list (one array per axis)"""
    coords = np.asarray(coords, dtype=np.float64)
    n, d = coords.shape
    ptr, _ = lists_to_csr(thresholds)
    thr = _f64(np.concatenate([np.asarray(t, dtype=np.float64) for t in thresholds]) if ptr[-1] else np.zeros(0))
    cm = _colmajor(coords)
    out = np.zeros(n * d)
    rc = lib.st_part_axis_parallel_lmt(_dp(cm), n, d, _dp(thr), _ip(ptr), _dp(out))
    if rc:
        raise SpamTreeError(rc, "st_part_axis_parallel_lmt")
    return out.reshape(d, n).T.copy()


def number_revalue(original_mat, from_val, to_val):
    """tree_dep.cpp:240-259"""
    om = np.asarray(original_mat, dtype=np.int64)
    nr, nc = om.shape
    flat = _i64(om.T.reshape(-1))
    fv, tv = _i64(from_val), _i64(to_val)
    out = np.zeros(nr * nc, dtype=np.int64)
    rc = lib.st_number_revalue(_ip(flat), nr, nc, _ip(fv), _ip(tv), fv.size, _ip(out))
    if rc:
        raise SpamTreeError(rc, "st_number_revalue")
    return out.reshape(nc, nr).T.copy()


def _make_edges(parchimat, non_empty_blocks, res_is_ref, limited):
    pm = np.asarray(parchimat, dtype=np.float64)
    nr, L = pm.shape
    flat = _colmajor(pm)
    ne, rr = _i64(non_empty_blocks), _i64(res_is_ref)
    counts = np.zeros(3, dtype=np.int64)
    rc = lib.st_make_edges(_dp(flat), nr, L, _ip(ne), ne.size, _ip(rr), int(limited), None, None, None, None, _ip(counts))
    if rc:
        raise SpamTreeError(rc, "st_make_edges")
    nb = int(counts[0])
    pp, pi = np.zeros(nb + 1, np.int64), np.zeros(max(int(counts[1]), 1), np.int64)
    cp, ci = np.zeros(nb + 1, np.int64), np.zeros(max(int(counts[2]), 1), np.int64)
    rc = lib.st_make_edges(_dp(flat), nr, L, _ip(ne), ne.size, _ip(rr), int(limited), _ip(pp), _ip(pi), _ip(cp), _ip(ci), _ip(counts))
    if rc:
        raise SpamTreeError(rc, "st_make_edges")
    return {"parents": csr_to_lists(pp, pi), "children": csr_to_lists(cp, ci)}


def make_edges(parchimat, non_empty_blocks, res_is_ref):
    """tree_dep.cpp:75-130 (parchimat: NaN = NA, 1-based block names; returned ids are 0-based like the reference)"""
    return _make_edges(parchimat, non_empty_blocks, res_is_ref, False)


def make_edges_limited(parchimat, non_empty_blocks, res_is_ref):
    """tree_dep.cpp:133-186"""
    return _make_edges(parchimat, non_empty_blocks, res_is_ref, True)


def _tree_attach(t, coords_new, mv_id_new, limited_tree):
    cn = _colmajor(np.asarray(coords_new, dtype=np.float64).reshape(-1, 2))
    nn = cn.size // 2
    mv = _i64(np.ones(nn, np.int64) if mv_id_new is None else mv_id_new).reshape(-1)
    if mv.size != nn:
        raise SpamTreeError(1, "mv_id_new must have one entry per row of coords_new")
    counts = np.zeros(2, dtype=np.int64)
    rc = lib.st_tree_attach(t, nn, _dp(cn), _ip(mv), int(bool(limited_tree)), None, None, None, _ip(counts))
    if rc:
        raise SpamTreeError(rc, lib.st_last_error(None).decode())
    group, pp = np.zeros(nn, np.int64), np.zeros(int(counts[0]) + 1, np.int64)
    pi = np.zeros(max(int(counts[1]), 1), np.int64)
    rc = lib.st_tree_attach(t, nn, _dp(cn), _ip(mv), int(bool(limited_tree)), _ip(group), _ip(pp), _ip(pi), _ip(counts))
    if rc:
        raise SpamTreeError(rc, lib.st_last_error(None).decode())
    return {"group": group, "parents_ptr": pp, "parents_idx": pi[:int(counts[1])], "n_groups": int(counts[0])}


def make_tree(coords, y, mv_id, cell_size=25, K=(2, 2), start_level=0, tree_depth=np.inf, last_not_reference=True,
              cherrypick_same_margin=True, cherrypick_group_locations=True, seed=0, *, coords_new=None, mv_id_new=None,
              limited_tree=False):
    """Deterministic stand-in for R's make_tree() + the graph-building tail of spamtree() (R/make_tree.R:1-420,
    R/spamtree_fit.R:288-324).  `coords` must be sorted by (Var1, Var2).  Returns the C++-boundary inputs.

    coords_new (n_new x 2, any order) and mv_id_new (1-based, default 1): new rows attached to the built tree by the rule of
    its prediction level (st_tree_attach), returned under "new": "group" (0-based group of each new row) and the parent CSR
    of the groups ("parents_ptr", "parents_idx": 0-based block ids, root first; limited_tree: the direct parent only).
    The tree itself does not depend on them."""
    coords = np.asarray(coords, dtype=np.float64)
    n = coords.shape[0]
    cm, yy, mv = _colmajor(coords), _f64(y).reshape(-1), _i64(mv_id).reshape(-1)
    o = _lib.StTreeOpts()
    o.n_all = n
    o.coords, o.y, o.mv_id = _dp(cm), _dp(yy), _ip(mv)
    o.cell_size = int(cell_size)
    o.K[0], o.K[1] = int(K[0]), int(K[1])
    o.start_level = int(start_level)
    o.tree_depth = 0 if not np.isfinite(tree_depth) else int(tree_depth)
    o.last_not_reference = int(bool(last_not_reference))
    o.cherrypick_same_margin = int(bool(cherrypick_same_margin))
    o.cherrypick_group_locations = int(bool(cherrypick_group_locations))
    o.seed = int(seed)
    t = C.c_void_p()
    rc = lib.st_make_tree(C.byref(o), C.byref(t))
    if rc:
        raise SpamTreeError(rc, lib.st_last_error(None).decode())
    try:
        sz = np.zeros(6, dtype=np.int64)
        lib.st_tree_sizes(t, _ip(sz))
        nb, nres, pr, pc, npar, nchi = [int(v) for v in sz]
        blocking, res = np.zeros(n, np.int64), np.zeros(n, np.int64)
        res_is_ref = np.zeros(nres, np.int64)
        parchi = np.zeros(pr * pc)
        ip_, ii = np.zeros(nb + 1, np.int64), np.zeros(n, np.int64)
        pp, pi = np.zeros(nb + 1, np.int64), np.zeros(max(npar, 1), np.int64)
        cp, ci = np.zeros(nb + 1, np.int64), np.zeros(max(nchi, 1), np.int64)
        bn, bg = np.zeros(nb), np.zeros(nb)
        lib.st_tree_get(t, _ip(blocking), _ip(res), _ip(res_is_ref), _dp(parchi), _ip(ip_), _ip(ii), _ip(pp), _ip(pi),
                        _ip(cp), _ip(ci), _dp(bn), _dp(bg))
        new = None if coords_new is None else _tree_attach(t, coords_new, mv_id_new, limited_tree)
    finally:
        lib.st_tree_destroy(t)
    out = {
        "blocking": blocking, "res": res, "res_is_ref": res_is_ref,
        "parchi_map": parchi.reshape(pc, pr).T.copy(),
        "indexing_ptr": ip_, "indexing_idx": ii, "parents_ptr": pp, "parents_idx": pi[:npar],
        "children_ptr": cp, "children_idx": ci[:nchi], "block_names": bn, "block_groups": bg, "n_blocks": nb,
    }
    if new is not None:
        out["new"] = new
    return out


def limited_edges_csr(tree, y):
    """(parents_ptr, parents_idx, children_ptr, children_idx) of make_edges_limited (tree_dep.cpp:133-186) for a tree
    returned by make_tree; y decides which blocks are non-empty (R/spamtree_fit.R:299-303)"""
    ne = np.unique(tree["blocking"][np.isfinite(np.asarray(y, dtype=np.float64).reshape(-1))])
    e = make_edges_limited(tree["parchi_map"], ne, tree["res_is_ref"])
    out = []
    for lists in (e["parents"], e["children"]):
        ptr = np.zeros(len(lists) + 1, dtype=np.int64)
        ptr[1:] = np.cumsum([len(a) for a in lists])
        idx = np.concatenate([np.asarray(a, dtype=np.int64) for a in lists]) if ptr[-1] else np.zeros(0, dtype=np.int64)
        out += [ptr, idx]
    return tuple(out)


def CrossCovarianceAG10(coords1, mv1, coords2, mv2, ai1, ai2, phi_i, thetamv, Dmat, device=0):
    """covariance_functions.cpp:301-355 (R export), evaluated on the GPU"""
    c1, c2 = np.asarray(coords1, dtype=np.float64), np.asarray(coords2, dtype=np.float64)
    n1, n2 = c1.shape[0], c2.shape[0]
    Dm = np.asarray(Dmat, dtype=np.float64)
    q = Dm.shape[1] if Dm.ndim == 2 else 1
    a, b, m1, m2 = _colmajor(c1), _colmajor(c2), _i64(mv1), _i64(mv2)
    A1, A2, PH, TM, DD = _f64(ai1), _f64(ai2), _f64(phi_i), _f64(np.atleast_1d(thetamv)), _colmajor(Dm)
    out = np.zeros(n1 * n2)
    rc = lib.st_cross_covariance_ag10(_dp(a), _ip(m1), n1, _dp(b), _ip(m2), n2, _dp(A1), _dp(A2), _dp(PH), _dp(TM), TM.size,
                                      _dp(DD), q, device, _dp(out))
    if rc:
        raise SpamTreeError(rc, lib.st_last_error(None).decode())
    return out.reshape(n2, n1).T.copy()


# --------------------------------------------------------------------------------------------- mh_adapt.h / mh_adapt.cpp
def par_huvtransf_fwd(par, set_unif_bounds):
    """mh_adapt.cpp:3-8"""
    a, b = _f64(par), _colmajor(np.asarray(set_unif_bounds, dtype=np.float64))
    out = np.zeros(a.size)
    rc = lib.st_par_huvtransf_fwd(_dp(a), a.size, _dp(b), _dp(out))
    if rc:
        raise SpamTreeError(rc, "st_par_huvtransf_fwd")
    return out


def par_huvtransf_back(par, set_unif_bounds):
    """mh_adapt.cpp:10-15"""
    a, b = _f64(par), _colmajor(np.asarray(set_unif_bounds, dtype=np.float64))
    out = np.zeros(a.size)
    rc = lib.st_par_huvtransf_back(_dp(a), a.size, _dp(b), _dp(out))
    if rc:
        raise SpamTreeError(rc, "st_par_huvtransf_back")
    return out


def mh_propose(param, set_unif_bounds, paramsd, U):
    """spamtree_fit.cpp:211-215 + calc_jacobian (mh_adapt.h:230-239): (new_param, jacobian, out_unif_bounds)"""
    a, b, sd, u = _f64(param), _colmajor(np.asarray(set_unif_bounds, dtype=np.float64)), _colmajor(np.asarray(paramsd, dtype=np.float64)), _f64(U)
    out = np.zeros(a.size + 2)
    rc = lib.st_mh_propose(a.size, _dp(a), _dp(b), _dp(sd), _dp(u), _dp(out))
    if rc:
        raise SpamTreeError(rc, "st_mh_propose")
    return out[:a.size].copy(), float(out[a.size]), bool(out[a.size + 1])


def do_I_accept(logaccept, u):
    """mh_adapt.h:20-36 with the caller's uniform draw"""
    return bool(lib.st_do_i_accept(float(logaccept), float(u)))


def ram_adapt(metropolis_sd, U, alpha):
    """class RAMAdapt (mh_adapt.h:40-135) over a recorded sequence: U steps x npar, alpha (steps).
    Returns (paramsd after the last step, trace steps x npar x npar)."""
    U = np.asarray(U, dtype=np.float64)
    steps, npar = U.shape
    sd, uu, al = _colmajor(np.asarray(metropolis_sd, dtype=np.float64)), _f64(U.reshape(-1)), _f64(alpha)
    out, tr = np.zeros(npar * npar), np.zeros(max(steps, 1) * npar * npar)
    rc = lib.st_ram_adapt(npar, _dp(sd), steps, _dp(uu), _dp(al), _dp(out), _dp(tr))
    if rc:
        raise SpamTreeError(rc, "st_ram_adapt: metropolis_sd is not positive definite")
    return out.reshape(npar, npar).T.copy(), tr[:steps * npar * npar].reshape(steps, npar, npar).transpose(0, 2, 1).copy()


# --------------------------------------------------------------------------------------------- the model layer
class SpamTreeMV:
    """src/spamtree_model.h:22-212.  Constructor arguments follow spamtree_model.cpp:8-37 (lists are 0-based id lists)."""

    def __init__(self, y, X, coords, mv_id, res_is_ref, parents, children, limited_tree, block_names, block_groups,
                 indexing, beta, theta, tausq, device=0, keep_H=True, smem_panel_bytes=0, csr=None, partition=None,
                 q=None):
        self.y = _f64(y).reshape(-1)
        self.n_all = self.y.size
        Xa = np.asarray(X, dtype=np.float64).reshape(self.n_all, -1)
        self.p = Xa.shape[1]
        self.mv_id = _i64(mv_id).reshape(-1)
        self.q = int(np.unique(self.mv_id).size) if q is None else int(q)
        self._X, self._coords = _colmajor(Xa), _colmajor(np.asarray(coords, dtype=np.float64))
        if csr is not None:
            ip_, ii, pp, pi, cp, ci = [_i64(a) for a in csr]
        else:
            ip_, ii = lists_to_csr(indexing)
            pp, pi = lists_to_csr(parents)
            cp, ci = lists_to_csr(children)
        self._csr = (ip_, ii, pp, pi, cp, ci)
        self.n_blocks = ip_.size - 1
        self._bn, self._bg, self._rr = _f64(block_names), _f64(block_groups), _i64(res_is_ref)
        self._theta, self._beta = _f64(theta), _f64(beta)
        self.npar = self._theta.size
        pr = _lib.StProblem()
        pr.n_all, pr.p, pr.q = self.n_all, self.p, self.q
        pr.y, pr.X, pr.coords, pr.mv_id = _dp(self.y), _dp(self._X), _dp(self._coords), _ip(self.mv_id)
        pr.n_blocks = self.n_blocks
        pr.indexing_ptr, pr.indexing_idx = _ip(ip_), _ip(ii)
        pr.parents_ptr, pr.parents_idx = _ip(pp), _ip(pi)
        pr.children_ptr, pr.children_idx = _ip(cp), _ip(ci)
        pr.block_names, pr.block_groups = _dp(self._bn), _dp(self._bg)
        pr.res_is_ref, pr.n_res = _ip(self._rr), self._rr.size
        pr.limited_tree = int(bool(limited_tree))
        pr.theta, pr.n_theta = _dp(self._theta), self.npar
        pr.beta, pr.tausq = _dp(self._beta), float(tausq)
        pr.device, pr.keep_H, pr.smem_panel_bytes = int(device), int(bool(keep_H)), int(smem_panel_bytes)
        if partition is not None and partition["nranks"] > 1:
            # partition: a sub-problem dict from spamtree_b200.partition.subproblem plus "allreduce": callable(ptr, count)
            fn = partition["allreduce"]

            def _cb(ctx, ptr, count):
                try:
                    fn(ptr, count)
                    return 0
                except Exception as ex:  # never let an exception cross the C boundary
                    print(f"spamtree_b200: allreduce callback failed: {ex}", flush=True)
                    return 1

            self._cb = _lib.ALLREDUCE_FN(_cb)
            self._grows = _i64(partition["global_rows"])
            pt = _lib.StPartition()
            pt.rank, pt.nranks, pt.n_top_levels = int(partition["rank"]), int(partition["nranks"]), int(partition["n_top_levels"])
            pt.rng_row_offset, pt.n_global_rows = int(partition["rng_row_offset"]), int(partition["n_global_rows"])
            pt.global_rows, pt.allreduce, pt.ctx = _ip(self._grows), self._cb, None
            self._pt = pt
            pr.partition = C.pointer(pt)
        h = C.c_void_p()
        rc = lib.st_create(C.byref(pr), C.byref(h))
        if rc:
            raise SpamTreeError(rc, lib.st_last_error(None).decode())
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            lib.st_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def _chk(self, rc):
        if rc:
            raise SpamTreeError(rc, lib.st_last_error(self._h).decode())

    # -- reference-named operations (slot 0 = param_data, 1 = alter_data)
    def theta_update(self, slot, theta):
        t = _f64(theta)
        self._chk(lib.st_theta_update(self._h, slot, _dp(t)))

    def get_loglik_comps_w(self, slot):
        """returns (acceptable, loglik_w, logdetCi)"""
        o = np.zeros(3)
        self._chk(lib.st_get_loglik_comps_w(self._h, slot, _dp(o)))
        return bool(o[2]), float(o[0]), float(o[1])

    def deal_with_w(self, z=None, seed=0):
        zz = None if z is None else _f64(z).reshape(-1)
        self._chk(lib.st_deal_with_w(self._h, _dp(zz), int(seed)))

    def get_loglik_w(self, slot=0):
        o = np.zeros(2)
        self._chk(lib.st_get_loglik_w(self._h, slot, _dp(o)))
        return float(o[0]), float(o[1])

    def accept_make_change(self):
        self._chk(lib.st_accept_make_change(self._h))

    def predict(self, theta_changed=True):
        self._chk(lib.st_predict(self._h, int(bool(theta_changed))))

    def gibbs_sample_beta(self, zb=None, faithful_index=True):
        z = None if zb is None else _colmajor(np.asarray(zb, dtype=np.float64))
        self._chk(lib.st_gibbs_sample_beta(self._h, _dp(z), int(bool(faithful_index))))

    def gibbs_sample_tausq(self, fixed=None):
        f = None if fixed is None else _f64(fixed)
        self._chk(lib.st_gibbs_sample_tausq(self._h, _dp(f)))

    def seed(self, s):
        self._chk(lib.st_seed(self._h, int(s)))

    # -- public fields
    @property
    def w(self):
        o = np.zeros(self.n_all)
        self._chk(lib.st_get_w(self._h, _dp(o)))
        return o

    @w.setter
    def w(self, v):
        a = _f64(v).reshape(-1)
        self._chk(lib.st_set_w(self._h, _dp(a)))

    def params(self):
        B, t, xb = np.zeros(self.p * self.q), np.zeros(self.q), np.zeros(self.n_all)
        self._chk(lib.st_get_params(self._h, _dp(B), _dp(t), _dp(xb)))
        return {"Bcoeff": B.reshape(self.q, self.p).T.copy(), "tausq_inv": t, "XB": xb}

    def set_tausq_inv(self, t):
        a = _f64(t)
        self._chk(lib.st_set_tausq_inv(self._h, _dp(a)))

    def node_state(self, which, u=0, slot=0):
        cnt = C.c_int64(0)
        self._chk(lib.st_get_node_state(self._h, slot, int(u), which.encode(), None, 0, C.byref(cnt)))
        o = np.zeros(max(cnt.value, 1))
        self._chk(lib.st_get_node_state(self._h, slot, int(u), which.encode(), _dp(o), o.size, C.byref(cnt)))
        return o[:cnt.value]

    def index(self, which, u=0, c=0):
        cnt = C.c_int64(0)
        self._chk(lib.st_get_index(self._h, which.encode(), int(u), int(c), None, 0, C.byref(cnt)))
        o = np.zeros(max(cnt.value, 1), dtype=np.int64)
        self._chk(lib.st_get_index(self._h, which.encode(), int(u), int(c), _ip(o), o.size, C.byref(cnt)))
        return o[:cnt.value]

    def predict_new(self, coords_new, X_new, mv_id_new, new_tree, samples=None, *, seed=1, draws=True, moments=False, z=None,
                    eps=None, keep_draws=False):
        """Posterior predictive draws at new locations from saved samples, without refitting (st_predict_new).

        coords_new (n_new x 2), X_new (n_new x p or None: no covariates), mv_id_new (1-based, None: all 1) in the caller's
        order; new_tree: the "new" entry of make_tree(..., coords_new=...) for the same rows (groups and their parents);
        samples: the dict mcmc() returns, or a subset of its sample columns ("theta_mcmc", "beta_mcmc", "tausq_mcmc",
        "w_mcmc").  z / eps (n_new x S): the normals of the w / y draws instead of the device's Philox streams.
        Returns the per-row summaries over the samples ("w_new_mean", "w_new_sd", "yhat_new_mean", "yhat_new_sd", sd with
        ddof = 1), "n_builds" and, with draws, "w_new" / "yhat_new" (n_new x S); with moments, the conditional "mean" /
        "sd" of every sample (n_new x S).

        samples=None: from every saved iteration of the last run of this handle with device_samples including "w"
        (st_predict_new_stored): the same outputs as from that run's host arrays, without them; normals from the device.
        keep_draws (samples=None only): the w_new / yhat_new draws also stay on the device for summarize("w_new" / "yhat_new")."""
        cn = np.asarray(coords_new, dtype=np.float64).reshape(-1, 2)
        nn = cn.shape[0]
        cm = _colmajor(cn)
        mv = _i64(np.ones(nn, np.int64) if mv_id_new is None else mv_id_new).reshape(-1)
        Xn = None if X_new is None else _colmajor(np.asarray(X_new, dtype=np.float64).reshape(nn, self.p))
        grp, pp, pi = _i64(new_tree["group"]), _i64(new_tree["parents_ptr"]), _i64(new_tree["parents_idx"])
        if mv.size != nn or grp.size != nn:
            raise SpamTreeError(1, "mv_id_new and new_tree['group'] must have one entry per new row")
        if samples is None:
            return self._predict_new_stored(cm, mv, Xn, grp, pp, pi, nn, seed, draws, moments, z, eps, keep_draws)
        if keep_draws:
            raise SpamTreeError(1, "keep_draws needs samples=None: draws are kept on the device only for a prediction from the "
                                   "device store")
        th = np.asarray(samples["theta_mcmc"], dtype=np.float64).reshape(self.npar, -1)
        S = th.shape[1]
        be = np.asarray(samples["beta_mcmc"], dtype=np.float64).reshape(self.p, S, self.q)
        ta = np.asarray(samples["tausq_mcmc"], dtype=np.float64).reshape(self.q, S)
        w = np.asarray(samples["w_mcmc"], dtype=np.float64).reshape(self.n_all, S)
        if not (w.flags.c_contiguous or w.flags.f_contiguous):
            w = np.ascontiguousarray(w)
        rs, ss = (S, 1) if w.flags.c_contiguous else (1, self.n_all)
        thf, bef, taf = [_f64(np.ravel(a, order="F")) for a in (th, be, ta)]
        zf = None if z is None else _f64(np.ravel(np.asarray(z, dtype=np.float64).reshape(nn, S), order="F"))
        ef = None if eps is None else _f64(np.ravel(np.asarray(eps, dtype=np.float64).reshape(nn, S), order="F"))
        sm = _lib.StPredSamples()
        sm.n_samples, sm.theta, sm.beta, sm.tausq = S, _dp(thf), _dp(bef), _dp(taf)
        sm.w, sm.w_row_stride, sm.w_sample_stride = w.ctypes.data_as(_lib.c_double_p), rs, ss
        sm.z, sm.eps, sm.seed = _dp(zf), _dp(ef), int(seed)
        return self._predict(cm, mv, Xn, grp, pp, pi, nn, S, draws, moments,
                             lambda r, o: lib.st_predict_new(self._h, r, C.byref(sm), o))

    def _predict_new_stored(self, cm, mv, Xn, grp, pp, pi, nn, seed, draws, moments, z, eps, keep_draws):
        if z is not None or eps is not None:
            raise SpamTreeError(1, "z / eps need host samples: a prediction from the device store draws its normals on the device")
        return self._predict(cm, mv, Xn, grp, pp, pi, nn, self._stored("w")[1], draws, moments,
                             lambda r, o: lib.st_predict_new_stored(self._h, r, int(seed), int(bool(keep_draws)), o))

    def _predict(self, cm, mv, Xn, grp, pp, pi, nn, S, draws, moments, call):
        """the new rows and the outputs of S samples for call(rows, out) -> status (st_predict_new or st_predict_new_stored)"""
        r = _lib.StNewRows()
        r.n_new, r.coords, r.mv_id, r.X = nn, _dp(cm), _ip(mv), _dp(Xn)
        r.n_groups, r.group, r.parents_ptr, r.parents_idx = pp.size - 1, _ip(grp), _ip(pp), _ip(pi)
        res = {k: np.zeros(nn) for k in ("w_new_mean", "w_new_sd", "yhat_new_mean", "yhat_new_sd")}
        dr = {k: np.zeros((S, nn)) for k in (("w_new", "yhat_new") if draws else ()) + (("mean", "sd") if moments else ())}
        o = _lib.StPredOut()
        o.w_new, o.y_new, o.mean, o.sd = [_dp(dr.get(k)) for k in ("w_new", "yhat_new", "mean", "sd")]
        o.w_mean, o.w_sd, o.y_mean, o.y_sd = [_dp(res[k]) for k in ("w_new_mean", "w_new_sd", "yhat_new_mean", "yhat_new_sd")]
        self._chk(call(C.byref(r), C.byref(o)))
        res.update({k: v.T for k, v in dr.items()})  # n_new x S (column-major views of the ABI's layout)
        res["n_builds"] = int(o.n_builds)
        return res

    _SUMMARY_WHICH = {"w": 0, "yhat": 1, "w_new": 2, "yhat_new": 3}

    def _stored(self, which):
        """(rows, draws) of a stored quantity; (0, 0) when nothing is stored"""
        o = _lib.StSummaryOut()
        if lib.st_summarize(self._h, self._SUMMARY_WHICH[which], None, 0, C.byref(o)):
            return 0, 0
        return int(o.n_rows), int(o.n_samples)

    def summarize(self, which, probs=(0.025, 0.5, 0.975)):
        """Per-row summaries of draws kept on the device (st_summarize): which = "w" / "yhat" of the last run with
        device_samples, "w_new" / "yhat_new" of the last predict_new(samples=None, keep_draws=True).  Returns "mean", "sd"
        (ddof = 1), "quantiles" (n x len(probs), numpy.quantile's "linear" method), "mcse" and "ess" (batch means) and "probs";
        rows in the order of w_mcmc / yhat_mcmc (boundary order) or of the new locations."""
        if which not in self._SUMMARY_WHICH:
            raise SpamTreeError(1, f"summarize: which must be one of {sorted(self._SUMMARY_WHICH)}")
        pr = _f64(np.atleast_1d(np.asarray(probs, dtype=np.float64)).reshape(-1))
        o = _lib.StSummaryOut()
        self._chk(lib.st_summarize(self._h, self._SUMMARY_WHICH[which], _dp(pr), pr.size, C.byref(o)))
        n = int(o.n_rows)
        res = {k: np.zeros(n) for k in ("mean", "sd", "mcse", "ess")}
        qt = np.zeros(n * pr.size)
        o.mean, o.sd, o.mcse, o.ess = [_dp(res[k]) for k in ("mean", "sd", "mcse", "ess")]
        o.quantiles = _dp(qt)
        self._chk(lib.st_summarize(self._h, self._SUMMARY_WHICH[which], _dp(pr), pr.size, C.byref(o)))
        res["quantiles"] = qt.reshape(pr.size, n).T.copy()
        res["probs"] = pr.copy()
        return res

    def fit_criteria(self, r_eff=1.0, integrated=False):
        """PSIS-LOO (with Pareto k-hat), WAIC and DIC per observation of the last run with device_samples including "w"
        (st_fit_criteria), from the draws of w kept on the device and that run's beta / tausq samples.  The log-likelihood is
        conditional on w: ll[i, s] = log N(y_i; x_i' beta_s[:, j] + w[i, s], tausq_s[j]), j the row's outcome.  Returns the
        per-row arrays "lpd", "elpd_loo", "p_loo", "pareto_k", "elpd_waic", "p_waic" (rows in boundary order, NaN where y is
        missing) and the totals of fit_criteria_loglik.

        With one latent w_i per observation, w_i is informed mostly by y_i itself, so PSIS-LOO of this model often shows
        k-hat > 0.7 on many rows (Vehtari et al. 2016): check "n_k_high" before relying on "elpd_loo".

        integrated=True: the same from the integrated log-likelihood of the last run with device_samples including
        "loglik_int" (st_fit_criteria_integrated, DESIGN.md §5f), in which w_i is integrated out of row i's term:
        ll[i, s] = log N(y_i - x_i' beta_s[:, j]; m_i, v_i + tausq_s[j]), N(m_i, v_i) the prior conditional of w_i given the
        rest of w, as the Gibbs sweep of draw s has it.  The DIC totals are NaN."""
        return _criteria([self], r_eff, integrated)

    def loglik_int(self):
        """The integrated log-likelihood of every row (boundary order, NaN where y is missing) from the last sweep that formed
        it (st_get_loglik_int): the last saved iteration of an mcmc call with device_samples including "loglik_int", or a
        deal_with_w while that call's store mask is set."""
        o = np.zeros(self.n_all)
        self._chk(lib.st_get_loglik_int(self._h, _dp(o)))
        return o

    _STORE_WHICH = {**_SUMMARY_WHICH, "loglik_int": 4}

    def stored_draws(self, which):
        """A host copy of the draws kept on the device (st_copy_store), (n_samples, n_rows): which = "w" / "yhat" /
        "loglik_int" of the last run with device_samples, "w_new" / "yhat_new" of the last predict_new(samples=None,
        keep_draws=True)."""
        if which not in self._STORE_WHICH:
            raise SpamTreeError(1, f"stored_draws: which must be one of {sorted(self._STORE_WHICH)}")
        k, n, S = self._STORE_WHICH[which], C.c_int64(0), C.c_int32(0)
        self._chk(lib.st_copy_store(self._h, k, None, C.byref(n), C.byref(S)))
        o = np.zeros((S.value, n.value))
        self._chk(lib.st_copy_store(self._h, k, _dp(o), C.byref(n), C.byref(S)))
        return o

    def bench_iteration(self, theta_prop, do_swap=False, seed=0):
        t, o, ms = _f64(theta_prop), np.zeros(3), np.zeros(6, dtype=np.float32)
        self._chk(lib.st_bench_iteration(self._h, _dp(t), int(bool(do_swap)), int(seed), _dp(o), ms.ctypes.data_as(_lib.c_float_p)))
        return o, ms

    def set_beta_index(self, faithful):
        """row index of the beta step in bench_iteration: the reference's (App. D #12) or the corrected one"""
        self._chk(lib.st_set_beta_index(self._h, int(bool(faithful))))

    def attach_nccl(self, unique_id):
        """collective over the ranks of the partition: the library creates its own NCCL communicator from the 128-byte id of
        st_nccl_unique_id and from then on enqueues its all-reduces on its stream (no callback, no host synchronisation)"""
        b = bytes(unique_id)
        assert len(b) == 128
        self._chk(lib.st_attach_nccl(self._h, b))

    def counters(self):
        o = np.zeros(8)
        self._chk(lib.st_get_counters(self._h, _dp(o)))
        return {"launches": o[0], "f_alg": o[1], "f_exec": o[2], "n_cov": o[3], "f_alg_build": o[4], "f_exec_build": o[5],
                "b_alg_build": o[6], "chain_state_bytes": o[7]}

    def sync(self):
        self._chk(lib.st_sync(self._h))

    def mcmc(self, set_unif_bounds, mcmcsd, keep, burn, thin, adapting=True, sample_beta=True, sample_tausq=True,
             sample_theta=True, sample_w=True, sample_predicts=True, faithful_beta_index=True, rng_mode=0, seed=1,
             save_w=True, save_yhat=True, device_samples=()):
        """the loop of spamtree_mv_mcmc (spamtree_fit.cpp:167-391).  device_samples: a subset of {"w", "yhat", "loglik_int"}
        whose saved draws stay on the device for summarize() and predict_new(samples=None) (rng_mode = 1); save_w / save_yhat
        still decide the host arrays.  "loglik_int": the integrated log-likelihood of every saved iteration, formed by its
        Gibbs sweep, for fit_criteria(integrated=True) and stored_draws("loglik_int") (needs sample_w)."""
        ds = set(device_samples or ())
        if not ds <= {"w", "yhat", "loglik_int"}:
            raise SpamTreeError(1, "device_samples must be a subset of {'w', 'yhat', 'loglik_int'}")
        self._chk(lib.st_keep_samples_on_device(self._h, (_lib.ST_KEEP_W if "w" in ds else 0) | (_lib.ST_KEEP_YHAT if "yhat" in ds else 0) |
                                                (_lib.ST_KEEP_LOGLIK_INT if "loglik_int" in ds else 0)))
        b, sd = _colmajor(np.asarray(set_unif_bounds, dtype=np.float64)), _colmajor(np.asarray(mcmcsd, dtype=np.float64))
        o = _lib.StMcmcOpts()
        o.set_unif_bounds, o.mcmcsd = _dp(b), _dp(sd)
        o.keep, o.burn, o.thin = int(keep), int(burn), int(thin)
        o.adapting, o.sample_beta, o.sample_tausq = int(adapting), int(sample_beta), int(sample_tausq)
        o.sample_theta, o.sample_w, o.sample_predicts = int(sample_theta), int(sample_w), int(sample_predicts)
        o.faithful_beta_index, o.rng_mode, o.seed = int(faithful_beta_index), int(rng_mode), int(seed)
        beta = np.zeros(self.p * keep * self.q)
        tausq, theta = np.zeros(self.q * keep), np.zeros(self.npar * keep)
        w = np.zeros(self.n_all * keep) if save_w else None
        yh = np.zeros(self.n_all * keep) if save_yhat else None
        psd = np.zeros(self.npar * self.npar)
        out = _lib.StMcmcOut()
        out.beta_mcmc, out.tausq_mcmc, out.theta_mcmc = _dp(beta), _dp(tausq), _dp(theta)
        out.w_mcmc, out.yhat_mcmc, out.paramsd = _dp(w), _dp(yh), _dp(psd)
        self._chk(lib.st_mcmc_run(self._h, C.byref(o), C.byref(out)))
        return {
            "w_mcmc": None if w is None else w.reshape(keep, self.n_all).T.copy(),
            "yhat_mcmc": None if yh is None else yh.reshape(keep, self.n_all).T.copy(),
            "beta_mcmc": beta.reshape(self.q, keep, self.p).transpose(2, 1, 0).copy(),  # p x keep x q
            "tausq_mcmc": tausq.reshape(keep, self.q).T.copy(),
            "theta_mcmc": theta.reshape(keep, self.npar).T.copy(),
            "paramsd": psd.reshape(self.npar, self.npar).T.copy(),
            "mcmc_time": out.mcmc_time, "n_accepted": out.n_accepted, "n_chol_fail": out.n_chol_fail,
        }


# --------------------------------------------------------------------------------------------- several chains (§5d)
def _chains_result(call, probs):
    """call(probs array, StChainsSummaryOut) -> status, made twice: for the sizes, then for the outputs"""
    pr = _f64(np.atleast_1d(np.asarray(probs, dtype=np.float64)).reshape(-1))
    o = _lib.StChainsSummaryOut()
    call(pr, o)
    n = int(o.n_rows)
    res = {k: np.zeros(n) for k in ("mean", "sd", "rhat", "ess_bulk", "ess_tail")}
    qt = np.zeros(n * pr.size)
    o.mean, o.sd, o.rhat, o.ess_bulk, o.ess_tail = [_dp(res[k]) for k in ("mean", "sd", "rhat", "ess_bulk", "ess_tail")]
    o.quantiles = _dp(qt)
    call(pr, o)
    res["quantiles"] = qt.reshape(pr.size, n).T.copy()
    res["probs"] = pr.copy()
    res["n_chains"], res["n_samples"] = int(o.n_chains), int(o.n_samples)
    return res


def summarize_chains(models, which, probs=(0.025, 0.5, 0.975)):
    """Pooled summaries and convergence diagnostics of the draws several chains keep on the device (st_summarize_chains):
    which = "w" / "yhat" of each model's last run with device_samples, or "w_new" / "yhat_new" of its last
    predict_new(samples=None, keep_draws=True).  The models must be on one device and store the same number of rows and
    draws; that they were built from the same problem is the caller's responsibility.  Returns per row "mean", "sd" (ddof 1)
    and "quantiles" (n x len(probs), numpy.quantile's "linear" method) over all chains' draws, rank-normalised split "rhat",
    "ess_bulk" and "ess_tail" (Vehtari et al. 2021, as ArviZ computes them; NaN below 4 draws per chain), and "probs",
    "n_chains", "n_samples".  R-hat can only detect what the chains' starting points expose: chains started from the same
    values that have not moved look converged to it."""
    if which not in SpamTreeMV._SUMMARY_WHICH:
        raise SpamTreeError(1, f"summarize_chains: which must be one of {sorted(SpamTreeMV._SUMMARY_WHICH)}")
    models = list(models)
    if not models:
        raise SpamTreeError(1, "summarize_chains: no models")
    hs = (C.c_void_p * len(models))(*[m._h for m in models])
    w = SpamTreeMV._SUMMARY_WHICH[which]

    def call(pr, o):
        models[0]._chk(lib.st_summarize_chains(hs, len(models), w, _dp(pr), pr.size, C.byref(o)))
    return _chains_result(call, probs)


def summarize_draws(draws, probs=(0.025, 0.5, 0.975), device=0):
    """summarize_chains on host draws (st_summarize_draws): draws (n_chains, n_samples, n_rows), or (n_chains, n_samples)
    for a scalar, are copied to the GPU for the call.  The same outputs, one row per trailing index.  The draws must be
    finite: a NaN or infinite draw is refused (SpamTreeError code 1)."""
    d = np.asarray(draws, dtype=np.float64)
    if d.ndim == 2:
        d = d[:, :, None]
    if d.ndim != 3:
        raise SpamTreeError(1, "summarize_draws: draws must be (n_chains, n_samples[, n_rows])")
    d = _f64(d)
    K, S, n = d.shape

    def call(pr, o):
        rc = lib.st_summarize_draws(int(device), _dp(d), n, K, S, _dp(pr), pr.size, C.byref(o))
        if rc:
            raise SpamTreeError(rc, lib.st_last_error(None).decode())
    return _chains_result(call, probs)


# --------------------------------------------------------------------------------------------- model criteria (§5e)
_CRIT_ROWS = ("lpd", "elpd_loo", "p_loo", "pareto_k", "elpd_waic", "p_waic")
_CRIT_TOTALS = ("elpd_loo_total", "se_elpd_loo", "p_loo_total", "looic", "se_looic", "elpd_waic_total", "se_elpd_waic",
                "p_waic_total", "waic", "se_waic", "lpd_total", "dbar", "dhat", "p_dic", "dic", "k_threshold")
_CRIT_COUNTS = ("n_rows", "n_obs", "n_k_high", "n_p_waic_high", "n_chains", "n_samples")


def _criteria_result(call):
    """call(StFitCriteriaOut) -> None (raising on a refusal), made twice: for the sizes, then for the outputs"""
    o = _lib.StFitCriteriaOut()
    call(o)
    n = int(o.n_rows)
    res = {k: np.zeros(n) for k in _CRIT_ROWS}
    for k in _CRIT_ROWS:
        setattr(o, k, _dp(res[k]))
    call(o)
    res.update({k: float(getattr(o, k)) for k in _CRIT_TOTALS})
    res.update({k: int(getattr(o, k)) for k in _CRIT_COUNTS})
    return res


def fit_criteria(models, r_eff=1.0, integrated=False):
    """PSIS-LOO, WAIC and DIC of the draws several chains of the same model keep on the device (st_fit_criteria): the w
    store of each model's last run with device_samples including "w", with that run's beta / tausq samples, pooled over
    the chains.  The models must be fits of the same data (y, X and mv_id are compared) with the same number of draws.

    Per row (rows in boundary order; NaN where y is missing): "lpd", "elpd_loo", "p_loo", "pareto_k" (the Pareto k-hat of
    PSIS, +inf when the tail is too short or constant), "elpd_waic", "p_waic" (ddof 1).  Totals over the observed rows:
    "elpd_loo_total", "se_elpd_loo", "p_loo_total", "looic", "se_looic", the same for WAIC, "lpd_total", DIC at the
    posterior means ("dbar", "dhat", "p_dic", "dic"), "k_threshold" (min(1 - 1 / log10(N), 0.7)), "n_k_high" (rows with
    k-hat above it), "n_p_waic_high" (rows with p_waic > 0.4), and "n_rows", "n_obs", "n_chains", "n_samples".  As R's loo
    package with one scalar r_eff (default 1) and gpdfit's weakly informative prior; DESIGN.md §5e has the definitions.

    The log-likelihood is conditional on w, one latent value per observation, so w_i is informed mostly by y_i itself and
    PSIS-LOO often shows k-hat > 0.7 on many rows (Vehtari, Mononen, Tolvanen, Sivula and Winther 2016): "n_k_high" says
    how far "elpd_loo" can be trusted.  Compare two fits of the same data with loo_compare.

    integrated=True: from each model's store of the integrated log-likelihood (device_samples including "loglik_int";
    st_fit_criteria_integrated, DESIGN.md §5f) instead, in which w_i is integrated out of row i's term: the same keys, with
    the DIC totals NaN."""
    return _criteria(models, r_eff, integrated)


def _criteria(models, r_eff, integrated=False):
    models = list(models)
    if not models:
        raise SpamTreeError(1, "fit_criteria: no models")
    hs = (C.c_void_p * len(models))(*[m._h for m in models])
    fn = lib.st_fit_criteria_integrated if integrated else lib.st_fit_criteria

    def call(o):
        models[0]._chk(fn(hs, len(models), float(r_eff), C.byref(o)))
    return _criteria_result(call)


def fit_criteria_loglik(loglik, r_eff=1.0, device=0):
    """The PSIS-LOO and WAIC part of fit_criteria on a log-likelihood the caller brings (st_fit_criteria_loglik): loglik
    (n_chains, n_samples, n_rows) or (n_samples, n_rows), copied to the GPU for the call.  A row of NaN is an unobserved
    row; any other NaN or infinite value is refused (SpamTreeError code 1).  The DIC totals are NaN."""
    d = np.asarray(loglik, dtype=np.float64)
    if d.ndim == 2:
        d = d[None]
    if d.ndim != 3:
        raise SpamTreeError(1, "fit_criteria_loglik: loglik must be (n_chains, n_samples, n_rows) or (n_samples, n_rows)")
    d = _f64(d)
    K, S, n = d.shape

    def call(o):
        rc = lib.st_fit_criteria_loglik(int(device), _dp(d), n, K, S, float(r_eff), C.byref(o))
        if rc:
            raise SpamTreeError(rc, lib.st_last_error(None).decode())
    return _criteria_result(call)


def loo_compare(a, b, criterion="elpd_loo"):
    """Difference of two fits of the same rows (results of fit_criteria / fit_criteria_loglik, or SpamTreeMV.fit_criteria):
    "elpd_diff" = sum_i (a_i - b_i) of the per-row criterion ("elpd_loo" or "elpd_waic") over the rows observed in both,
    "se_diff" = sqrt(n var(a_i - b_i, ddof 1)) and "n".  Positive: a predicts better.  spamtree() orders rows by their
    coordinates alone, so two of its fits of the same data share the row order."""
    if criterion not in ("elpd_loo", "elpd_waic"):
        raise SpamTreeError(1, "loo_compare: criterion must be 'elpd_loo' or 'elpd_waic'")
    x, z = np.asarray(a[criterion], dtype=np.float64), np.asarray(b[criterion], dtype=np.float64)
    if x.shape != z.shape:
        raise SpamTreeError(1, "loo_compare: the two results have different numbers of rows")
    dlt = (x - z)[~(np.isnan(x) | np.isnan(z))]
    n = dlt.size
    return {"elpd_diff": float(dlt.sum()), "se_diff": float(np.sqrt(n * np.var(dlt, ddof=1))) if n > 1 else float("nan"), "n": n}


def spamtree_mv_mcmc(y, X, Z, coords, mv_id, blocking, gix_block, res_is_ref, parents, children, limited_tree,
                     layer_names, layer_gibbs_group, indexing, set_unif_bounds_in, start_w, theta, beta, tausq, mcmcsd,
                     mcmc_keep=100, mcmc_burn=100, mcmc_thin=1, num_threads=1, use_alg='S', adapting=False,
                     main_verbose=True, verbose=False, debug=False, printall=False, sample_beta=True,
                     sample_tausq=True, sample_theta=True, sample_w=True, sample_predicts=True, *, device=0, seed=1,
                     rng_mode=0, csr=None, save_w=True, save_yhat=True, keep_H=False):
    """Mirror of the Rcpp export (src/spamtree_fit.cpp:5-54): same positional arguments, same returned names
    (:403-414).  Z, blocking, gix_block, start_w, num_threads, use_alg and the verbosity flags are accepted and ignored
    exactly as the reference ignores them (SURVEY App. D #6); keyword-only arguments are additions of this build."""
    model = SpamTreeMV(y, X, coords, mv_id, res_is_ref, parents, children, limited_tree, layer_names, layer_gibbs_group,
                       indexing, beta, theta, tausq, device=device, csr=csr, keep_H=keep_H)
    try:
        return _mv_mcmc_on(model, indexing, set_unif_bounds_in, mcmcsd, mcmc_keep, mcmc_burn, mcmc_thin, adapting, sample_beta,
                           sample_tausq, sample_theta, sample_w, sample_predicts, rng_mode, seed, save_w, save_yhat)
    finally:
        model.close()


def _mv_mcmc_on(model, indexing, set_unif_bounds_in, mcmcsd, mcmc_keep, mcmc_burn, mcmc_thin, adapting, sample_beta,
                sample_tausq, sample_theta, sample_w, sample_predicts, rng_mode, seed, save_w, save_yhat, device_samples=()):
    """the chain and the returned list of spamtree_mv_mcmc on an open handle (the caller closes it)"""
    res = model.mcmc(set_unif_bounds_in, mcmcsd, mcmc_keep, mcmc_burn, mcmc_thin, adapting, sample_beta,
                     sample_tausq, sample_theta, sample_w, sample_predicts, True, rng_mode, seed, save_w, save_yhat,
                     device_samples=device_samples)
    # the rest of the reference's returned list (spamtree_fit.cpp:410-412)
    res["block_ct_obs"] = model.index("block_ct_obs")
    res["indexing"] = indexing if indexing is not None else csr_to_lists(model._csr[0], model._csr[1])
    res["parents_indexing"] = [model.index("parents_indexing", u) for u in range(model.n_blocks)]
    return res


def spamtree(y, x, coords, mv_id=None, cell_size=25, K=None, start_level=0, tree_depth=np.inf, last_not_reference=True,
             limited_tree=False, cherrypick_same_margin=True, cherrypick_group_locations=True, mvbias=0,
             mcmc=None, num_threads=4, verbose=False, settings=None, prior=None, starting=None, debug=None, *,
             device=0, seed=1, rng_mode=1, tree_seed=0, coords_new=None, x_new=None, mv_id_new=None, summary_probs=None,
             n_chains=1, fit_criteria=False, loo_integrated=False):
    """Mirror of the R entry point spamtree() (R/spamtree_fit.R:1-371): same arguments and defaults, same returned
    names (`coords`, `coordsinfo`, `mv_id` + everything spamtree_mv_mcmc returns).  The tree is built by the
    deterministic stand-in for make_tree() (mvbias other than 0 is not supported).

    coords_new (n_new x 2), x_new (n_new x p, required with coords_new) and mv_id_new (1-based; None: all 1): locations to
    predict at after the fit, attached to the fitted tree without changing it (SpamTreeMV.predict_new from every saved
    sample, on the same handle).  The result then also holds "w_new_mcmc" and "yhat_new_mcmc" (n_new x keep, rows in the
    order given) and "w_new_mean", "w_new_sd", "yhat_new_mean", "yhat_new_sd" (n_new); every other key is what the call
    without coords_new returns.

    summary_probs (probabilities in [0, 1]): the draws of w and yhat (and of the new locations) stay on the device and are
    summarised there (SpamTreeMV.summarize): the result gains "w_summary" and "yhat_summary" (with coords_new also
    "w_new_summary" and "yhat_new_summary"), each a dict of per-row "mean", "sd", "quantiles" at summary_probs, "mcse",
    "ess" and "probs", and "w_mcmc" / "yhat_mcmc" (and "w_new_mcmc" / "yhat_new_mcmc") are None instead of host copies of
    every draw.  Needs rng_mode = 1.  Every other key is unchanged.

    n_chains = K > 1 (rng_mode = 1): K chains, chain k on its own handle with seed + k, one after another; starting may be
    a list of K dicts, one per chain, else every chain starts from the same values.  As in the single-chain call, only the
    "beta" and "tausq" starts are used (theta starts at the middle of its bounds and w at 0, as in the reference), so a
    per-chain dict that sets "theta" or "w" is refused rather than ignored.  The result holds "coords",
    "coordsinfo", "mv_id" and "chains", a list of K dicts, dict k being what spamtree(..., seed=seed + k) returns besides
    those three.  It also holds the pooled summaries and diagnostics of summarize_chains / summarize_draws at summary_probs
    (default (0.025, 0.5, 0.975)): "w_summary" and "yhat_summary" (with coords_new also "w_new_summary" and
    "yhat_new_summary"), and "theta_summary", "beta_summary" (rows in beta_mcmc's p x q order, column-major) and
    "tausq_summary" over the chains' samples.  R-hat can only detect what the starting points expose: identical starts are
    the default only because the reference has a single start, so pass dispersed beta / tausq starts to test convergence.

    fit_criteria=True (rng_mode = 1): the result gains "fit_criteria", PSIS-LOO, WAIC and DIC per observation and in total
    (the dict of SpamTreeMV.fit_criteria; with n_chains > 1 pooled over the chains), formed on the device from the draws of
    w.  Every other key is what the call without it returns.  Compare two fits of the same data with loo_compare.

    loo_integrated=True (rng_mode = 1): the result gains "fit_criteria_integrated", the same criteria from the integrated
    log-likelihood (SpamTreeMV.fit_criteria(integrated=True), DESIGN.md §5f; with n_chains > 1 pooled over the chains), in
    which w_i is integrated out of row i's term so that fewer rows have a high Pareto k-hat.  It has the keys of
    "fit_criteria", with the DIC totals NaN, so loo_compare takes it.  Every other key is what the call without it returns."""
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    x = np.asarray(x, dtype=np.float64).reshape(y.size, -1)
    coords = np.asarray(coords, dtype=np.float64)
    mv_id = np.ones(y.size, dtype=np.int64) if mv_id is None else np.asarray(mv_id, dtype=np.int64)
    K = (2,) * coords.shape[1] if K is None else K
    mcmc = {"keep": 1000, "burn": 0, "thin": 1, **(mcmc or {})}
    settings = {"adapting": True, "mcmcsd": .01, "debug": False, "printall": False, **(settings or {})}
    prior = {"set_unif_bounds": None, "btmlim": None, "toplim": None, "vlim": None, **(prior or {})}
    n_chains = int(n_chains)
    if n_chains < 1:
        raise SpamTreeError(1, "n_chains must be at least 1")
    if n_chains > 1 and rng_mode != 1:
        raise SpamTreeError(1, "n_chains > 1 needs rng_mode = 1: the pooled summaries read every chain's draws on the device")
    if fit_criteria and rng_mode != 1:
        raise SpamTreeError(1, "fit_criteria needs rng_mode = 1: the criteria read the draws of w kept on the device")
    if loo_integrated and rng_mode != 1:
        raise SpamTreeError(1, "loo_integrated needs rng_mode = 1: the criteria read the integrated log-likelihood kept on the device")
    crit, iloo = bool(fit_criteria), bool(loo_integrated)
    if isinstance(starting, (list, tuple)):
        if len(starting) != n_chains:
            raise SpamTreeError(1, "starting: one dict per chain")
        if any((st or {}).get(key) is not None for st in starting for key in ("theta", "w")):
            raise SpamTreeError(4, "starting: per-chain theta or w starts are not supported (theta starts at the middle of its "
                                   "bounds and w at 0, as in the reference); disperse beta and tausq instead")
        starts = [{"beta": None, "tausq": None, "theta": None, "w": None, **(st or {})} for st in starting]
    else:
        starts = [{"beta": None, "tausq": None, "theta": None, "w": None, **(starting or {})}] * n_chains
    starting = starts[0]
    debug = {"sample_beta": True, "sample_tausq": True, "sample_theta": True, "sample_w": True, "sample_predicts": True,
             **(debug or {})}
    if mvbias != 0:
        raise SpamTreeError(4, "mvbias != 0 is not supported by the deterministic tree builder")
    if coords_new is not None and x_new is None:  # (without it yhat_new would lack x' beta)
        raise SpamTreeError(1, "coords_new needs x_new: the covariates of the new locations (n_new x p)")
    dd, p = coords.shape[1], x.shape[1]
    if dd > 2:
        raise SpamTreeError(4, "Not implemented in domains of dimension d>2.")  # R/spamtree_fit.R:58-60
    q = int(np.unique(mv_id).size)
    k = q * (q - 1) // 2
    btmlim = 1e-3 if prior["btmlim"] is None else prior["btmlim"]
    toplim = 1e3 if prior["toplim"] is None else prior["toplim"]
    vlim = toplim if prior["vlim"] is None else prior["vlim"]
    n_cbase = 3 if q > 2 else 1
    npars = 3 * q + n_cbase
    bounds = np.zeros((npars, 2))  # :111-134
    bounds[:, 0], bounds[:, 1] = btmlim, toplim
    if q > 1:
        bounds[1:q, 0] = -toplim
    if n_cbase == 3:
        bounds[npars - 2, :] = (btmlim, 1 - btmlim)
    if q > 1:
        vb = np.zeros((k, 2))
        vb[:, 0], vb[:, 1] = btmlim, vlim - btmlim
        bounds = np.vstack([bounds, vb])
    start_theta = bounds.mean(axis=1)  # :138
    sd = settings["mcmcsd"]
    mcmc_mh_sd = np.eye(start_theta.size) * sd if np.ndim(sd) == 0 else np.asarray(sd, dtype=np.float64)
    # rows sorted by coordinates, ties by input order (:214, :267-269)
    ix = np.arange(y.size)
    order = np.lexsort((ix, coords[:, 1], coords[:, 0]))
    cs, ys, xs, mvs = coords[order], y[order], x[order], mv_id[order]
    tree = make_tree(cs, ys, mvs, cell_size, K, start_level, tree_depth, last_not_reference, cherrypick_same_margin,
                     cherrypick_group_locations, tree_seed, coords_new=coords_new, mv_id_new=mv_id_new,
                     limited_tree=limited_tree)
    Z = np.zeros((y.size, q))
    Z[np.arange(y.size), mvs - 1] = 1
    csr = (tree["indexing_ptr"], tree["indexing_idx"], tree["parents_ptr"], tree["parents_idx"], tree["children_ptr"],
           tree["children_idx"])
    if limited_tree:  # R/spamtree_fit.R:310-311: make_edges_limited on the same parent-child map
        csr = csr[:2] + limited_edges_csr(tree, ys)
    coordsinfo = {"Var1": cs[:, 0], "Var2": cs[:, 1], "ix": order + 1, "block": tree["blocking"], "res": tree["res"]}

    def open_chain(st):
        # (the arguments spamtree_mv_mcmc receives, R/spamtree_fit.R:327-362, on a handle that stays open for the prediction)
        sb = np.zeros(p) if st["beta"] is None else np.asarray(st["beta"], dtype=np.float64)
        stau = .1 if st["tausq"] is None else st["tausq"]
        return SpamTreeMV(ys, xs, cs, mvs, tree["res_is_ref"], None, None, limited_tree, tree["block_names"], tree["block_groups"],
                          None, sb, start_theta, stau, device=device, csr=csr, keep_H=False)

    summ = summary_probs is not None

    def run_chain(model, seed_k, on_device):
        """the chain and its prediction; on_device: the draws also stay on the device for the pooled summaries"""
        results = _mv_mcmc_on(model, None, bounds, mcmc_mh_sd, mcmc["keep"], mcmc["burn"], mcmc["thin"], settings["adapting"],
                              debug["sample_beta"], debug["sample_tausq"], debug["sample_theta"], debug["sample_w"],
                              debug["sample_predicts"], rng_mode, seed_k, not summ, not summ,
                              device_samples=(("w", "yhat") if summ or on_device else ("w",) if crit else ()) +
                              (("loglik_int",) if iloo else ()))
        if summ:
            results["w_summary"] = model.summarize("w", summary_probs)
            results["yhat_summary"] = model.summarize("yhat", summary_probs)
        if coords_new is not None:
            if summ or on_device:  # (the same draws as from the host samples: DESIGN.md §5c)
                pr = model.predict_new(coords_new, x_new, mv_id_new, tree["new"], None, seed=seed_k, draws=not summ, keep_draws=True)
            else:
                pr = model.predict_new(coords_new, x_new, mv_id_new, tree["new"], results, seed=seed_k)
            if summ:
                results["w_new_mcmc"] = results["yhat_new_mcmc"] = None
                results["w_new_summary"] = model.summarize("w_new", summary_probs)
                results["yhat_new_summary"] = model.summarize("yhat_new", summary_probs)
            else:
                results["w_new_mcmc"], results["yhat_new_mcmc"] = np.ascontiguousarray(pr["w_new"]), np.ascontiguousarray(pr["yhat_new"])
            for k in ("w_new_mean", "w_new_sd", "yhat_new_mean", "yhat_new_sd"):
                results[k] = pr[k]
        return results

    if n_chains == 1:
        model = open_chain(starting)
        try:
            results = run_chain(model, seed, False)
            if crit:
                results["fit_criteria"] = model.fit_criteria()
            if iloo:
                results["fit_criteria_integrated"] = model.fit_criteria(integrated=True)
        finally:
            model.close()
        return {"coords": cs, "coordsinfo": coordsinfo, "mv_id": mv_id, **results}
    models, chains = [], []
    probs = summary_probs if summ else (0.025, 0.5, 0.975)
    out = {"coords": cs, "coordsinfo": coordsinfo, "mv_id": mv_id, "chains": chains}
    try:
        for k in range(n_chains):  # every handle keeps its draws on the device until the pooled summaries are formed
            models.append(open_chain(starts[k]))
            chains.append(run_chain(models[-1], seed + k, True))
        for which in ("w", "yhat") + (("w_new", "yhat_new") if coords_new is not None else ()):
            out[which + "_summary"] = summarize_chains(models, which, probs)
        if crit:
            out["fit_criteria"] = _criteria(models, 1.0)
        if iloo:
            out["fit_criteria_integrated"] = _criteria(models, 1.0, integrated=True)
    finally:
        for m in models:
            m.close()
    out["theta_summary"] = summarize_draws(np.stack([c["theta_mcmc"].T for c in chains]), probs, device=device)
    out["beta_summary"] = summarize_draws(np.stack([c["beta_mcmc"].transpose(1, 2, 0).reshape(-1, p * q) for c in chains]),
                                          probs, device=device)
    out["tausq_summary"] = summarize_draws(np.stack([c["tausq_mcmc"].T for c in chains]), probs, device=device)
    return out
