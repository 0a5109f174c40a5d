"""ctypes loader for libspamtree_b200.so (the C ABI in include/spamtree_b200.h).

The product path has no CPU fallback: if the shared library is missing this module raises at import.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SPAMTREE_B200_LIB") or os.path.join(_HERE, "libspamtree_b200.so")  # (override: kernel-variant experiments)

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "or `make -C spamtree_b200/csrc` (there is no CPU fallback)")

lib = C.CDLL(LIB_PATH)

c_double_p = C.POINTER(C.c_double)
c_int64_p = C.POINTER(C.c_int64)
c_float_p = C.POINTER(C.c_float)


ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64)


class StPartition(C.Structure):
    _fields_ = [
        ("rank", C.c_int32), ("nranks", C.c_int32), ("n_top_levels", C.c_int32),
        ("rng_row_offset", C.c_int64), ("n_global_rows", C.c_int64), ("global_rows", c_int64_p),
        ("allreduce", ALLREDUCE_FN), ("ctx", C.c_void_p),
    ]


class StProblem(C.Structure):
    _fields_ = [
        ("n_all", C.c_int64), ("p", C.c_int32), ("q", C.c_int32),
        ("y", c_double_p), ("X", c_double_p), ("coords", c_double_p), ("mv_id", c_int64_p),
        ("n_blocks", C.c_int32),
        ("indexing_ptr", c_int64_p), ("indexing_idx", c_int64_p),
        ("parents_ptr", c_int64_p), ("parents_idx", c_int64_p),
        ("children_ptr", c_int64_p), ("children_idx", c_int64_p),
        ("block_names", c_double_p), ("block_groups", c_double_p),
        ("res_is_ref", c_int64_p), ("n_res", C.c_int32), ("limited_tree", C.c_int32),
        ("theta", c_double_p), ("n_theta", C.c_int32),
        ("beta", c_double_p), ("tausq", C.c_double),
        ("device", C.c_int32), ("keep_H", C.c_int32), ("smem_panel_bytes", C.c_int64),
        ("partition", C.POINTER(StPartition)),
    ]


class StMcmcOpts(C.Structure):
    _fields_ = [
        ("set_unif_bounds", c_double_p), ("mcmcsd", c_double_p),
        ("keep", C.c_int32), ("burn", C.c_int32), ("thin", C.c_int32),
        ("adapting", C.c_int32), ("sample_beta", C.c_int32), ("sample_tausq", C.c_int32),
        ("sample_theta", C.c_int32), ("sample_w", C.c_int32), ("sample_predicts", C.c_int32),
        ("faithful_beta_index", C.c_int32), ("rng_mode", C.c_int32), ("seed", C.c_uint64),
    ]


class StMcmcOut(C.Structure):
    _fields_ = [
        ("beta_mcmc", c_double_p), ("tausq_mcmc", c_double_p), ("theta_mcmc", c_double_p),
        ("w_mcmc", c_double_p), ("yhat_mcmc", c_double_p), ("paramsd", c_double_p),
        ("mcmc_time", C.c_double), ("n_accepted", C.c_int64), ("n_chol_fail", C.c_int64),
    ]


class StTreeOpts(C.Structure):
    _fields_ = [
        ("n_all", C.c_int64), ("coords", c_double_p), ("y", c_double_p), ("mv_id", c_int64_p),
        ("cell_size", C.c_int32), ("K", C.c_int32 * 2), ("start_level", C.c_int32), ("tree_depth", C.c_int32),
        ("last_not_reference", C.c_int32), ("cherrypick_same_margin", C.c_int32),
        ("cherrypick_group_locations", C.c_int32), ("seed", C.c_uint64),
    ]


class StNewRows(C.Structure):
    _fields_ = [
        ("n_new", C.c_int64), ("coords", c_double_p), ("mv_id", c_int64_p), ("X", c_double_p),
        ("n_groups", C.c_int64), ("group", c_int64_p), ("parents_ptr", c_int64_p), ("parents_idx", c_int64_p),
    ]


class StPredSamples(C.Structure):
    _fields_ = [
        ("n_samples", C.c_int32), ("theta", c_double_p), ("beta", c_double_p), ("tausq", c_double_p), ("w", c_double_p),
        ("w_row_stride", C.c_int64), ("w_sample_stride", C.c_int64), ("z", c_double_p), ("eps", c_double_p),
        ("seed", C.c_uint64),
    ]


class StPredOut(C.Structure):
    _fields_ = [
        ("w_new", c_double_p), ("y_new", c_double_p), ("mean", c_double_p), ("sd", c_double_p),
        ("w_mean", c_double_p), ("w_sd", c_double_p), ("y_mean", c_double_p), ("y_sd", c_double_p),
        ("n_builds", C.c_int64),
    ]


class StSummaryOut(C.Structure):
    _fields_ = [
        ("mean", c_double_p), ("sd", c_double_p), ("quantiles", c_double_p), ("mcse", c_double_p), ("ess", c_double_p),
        ("n_rows", C.c_int64), ("n_samples", C.c_int32),
    ]


class StChainsSummaryOut(C.Structure):
    _fields_ = [
        ("mean", c_double_p), ("sd", c_double_p), ("quantiles", c_double_p), ("rhat", c_double_p), ("ess_bulk", c_double_p),
        ("ess_tail", c_double_p), ("n_rows", C.c_int64), ("n_chains", C.c_int32), ("n_samples", C.c_int32),
    ]


class StFitCriteriaOut(C.Structure):
    _fields_ = [
        ("lpd", c_double_p), ("elpd_loo", c_double_p), ("p_loo", c_double_p), ("pareto_k", c_double_p),
        ("elpd_waic", c_double_p), ("p_waic", c_double_p),
        ("elpd_loo_total", C.c_double), ("se_elpd_loo", C.c_double), ("p_loo_total", C.c_double), ("looic", C.c_double),
        ("se_looic", C.c_double), ("elpd_waic_total", C.c_double), ("se_elpd_waic", C.c_double), ("p_waic_total", C.c_double),
        ("waic", C.c_double), ("se_waic", C.c_double), ("lpd_total", C.c_double),
        ("dbar", C.c_double), ("dhat", C.c_double), ("p_dic", C.c_double), ("dic", C.c_double), ("k_threshold", C.c_double),
        ("n_rows", C.c_int64), ("n_obs", C.c_int64), ("n_k_high", C.c_int64), ("n_p_waic_high", C.c_int64),
        ("n_chains", C.c_int32), ("n_samples", C.c_int32),
    ]


ST_KEEP_W, ST_KEEP_YHAT, ST_KEEP_LOGLIK_INT = 1, 2, 4


# every symbol include/spamtree_b200.h declares, with its signature
SIGNATURES = {
    "st_version": (C.c_char_p, []),
    "st_create": (C.c_int, [C.POINTER(StProblem), C.POINTER(C.c_void_p)]),
    "st_destroy": (None, [C.c_void_p]),
    "st_last_error": (C.c_char_p, [C.c_void_p]),
    "st_theta_update": (C.c_int, [C.c_void_p, C.c_int, c_double_p]),
    "st_get_loglik_comps_w": (C.c_int, [C.c_void_p, C.c_int, c_double_p]),
    "st_deal_with_w": (C.c_int, [C.c_void_p, c_double_p, C.c_uint64]),
    "st_get_loglik_w": (C.c_int, [C.c_void_p, C.c_int, c_double_p]),
    "st_accept_make_change": (C.c_int, [C.c_void_p]),
    "st_predict": (C.c_int, [C.c_void_p, C.c_int]),
    "st_gibbs_sample_beta": (C.c_int, [C.c_void_p, c_double_p, C.c_int]),
    "st_gibbs_sample_tausq": (C.c_int, [C.c_void_p, c_double_p]),
    "st_seed": (C.c_int, [C.c_void_p, C.c_uint64]),
    "st_get_w": (C.c_int, [C.c_void_p, c_double_p]),
    "st_set_w": (C.c_int, [C.c_void_p, c_double_p]),
    "st_get_params": (C.c_int, [C.c_void_p, c_double_p, c_double_p, c_double_p]),
    "st_set_tausq_inv": (C.c_int, [C.c_void_p, c_double_p]),
    "st_get_node_state": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_char_p, c_double_p, C.c_int64, c_int64_p]),
    "st_get_index": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.c_int, c_int64_p, C.c_int64, c_int64_p]),
    "st_mcmc_run": (C.c_int, [C.c_void_p, C.POINTER(StMcmcOpts), C.POINTER(StMcmcOut)]),
    "st_predict_new": (C.c_int, [C.c_void_p, C.POINTER(StNewRows), C.POINTER(StPredSamples), C.POINTER(StPredOut)]),
    "st_keep_samples_on_device": (C.c_int, [C.c_void_p, C.c_int32]),
    "st_get_loglik_int": (C.c_int, [C.c_void_p, c_double_p]),
    "st_copy_store": (C.c_int, [C.c_void_p, C.c_int32, c_double_p, c_int64_p, C.POINTER(C.c_int32)]),
    "st_summarize": (C.c_int, [C.c_void_p, C.c_int32, c_double_p, C.c_int32, C.POINTER(StSummaryOut)]),
    "st_predict_new_stored": (C.c_int, [C.c_void_p, C.POINTER(StNewRows), C.c_uint64, C.c_int32, C.POINTER(StPredOut)]),
    "st_summarize_chains": (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_int32, c_double_p, C.c_int32,
                                      C.POINTER(StChainsSummaryOut)]),
    "st_summarize_draws": (C.c_int, [C.c_int32, c_double_p, C.c_int64, C.c_int32, C.c_int32, c_double_p, C.c_int32,
                                     C.POINTER(StChainsSummaryOut)]),
    "st_fit_criteria": (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_double, C.POINTER(StFitCriteriaOut)]),
    "st_fit_criteria_integrated": (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_double, C.POINTER(StFitCriteriaOut)]),
    "st_fit_criteria_loglik": (C.c_int, [C.c_int32, c_double_p, C.c_int64, C.c_int32, C.c_int32, C.c_double,
                                         C.POINTER(StFitCriteriaOut)]),
    "st_bench_iteration": (C.c_int, [C.c_void_p, c_double_p, C.c_int, C.c_uint64, c_double_p, c_float_p]),
    "st_set_beta_index": (C.c_int, [C.c_void_p, C.c_int]),
    "st_get_counters": (C.c_int, [C.c_void_p, c_double_p]),
    "st_par_huvtransf_fwd": (C.c_int, [c_double_p, C.c_int32, c_double_p, c_double_p]),
    "st_par_huvtransf_back": (C.c_int, [c_double_p, C.c_int32, c_double_p, c_double_p]),
    "st_mh_propose": (C.c_int, [C.c_int32, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p]),
    "st_do_i_accept": (C.c_int, [C.c_double, C.c_double]),
    "st_ram_adapt": (C.c_int, [C.c_int32, c_double_p, C.c_int32, c_double_p, c_double_p, c_double_p, c_double_p]),
    "st_nccl_unique_id": (C.c_int, [C.c_char_p]),
    "st_attach_nccl": (C.c_int, [C.c_void_p, C.c_char_p]),
    "st_sync": (C.c_int, [C.c_void_p]),
    "st_kthresholds": (C.c_int, [c_double_p, C.c_int64, C.c_int32, c_double_p]),
    "st_part_axis_parallel_lmt": (C.c_int, [c_double_p, C.c_int64, C.c_int32, c_double_p, c_int64_p, c_double_p]),
    "st_number_revalue": (C.c_int, [c_int64_p, C.c_int64, C.c_int32, c_int64_p, c_int64_p, C.c_int64, c_int64_p]),
    "st_make_edges": (C.c_int, [c_double_p, C.c_int64, C.c_int32, c_int64_p, C.c_int64, c_int64_p, C.c_int32,
                                c_int64_p, c_int64_p, c_int64_p, c_int64_p, c_int64_p]),
    "st_make_tree": (C.c_int, [C.POINTER(StTreeOpts), C.POINTER(C.c_void_p)]),
    "st_tree_destroy": (None, [C.c_void_p]),
    "st_tree_sizes": (C.c_int, [C.c_void_p, c_int64_p]),
    "st_tree_get": (C.c_int, [C.c_void_p, c_int64_p, c_int64_p, c_int64_p, c_double_p, c_int64_p, c_int64_p,
                              c_int64_p, c_int64_p, c_int64_p, c_int64_p, c_double_p, c_double_p]),
    "st_tree_attach": (C.c_int, [C.c_void_p, C.c_int64, c_double_p, c_int64_p, C.c_int32, c_int64_p, c_int64_p,
                                 c_int64_p, c_int64_p]),
    "st_cross_covariance_ag10": (C.c_int, [c_double_p, c_int64_p, C.c_int64, c_double_p, c_int64_p, C.c_int64,
                                           c_double_p, c_double_p, c_double_p, c_double_p, C.c_int32, c_double_p,
                                           C.c_int32, C.c_int32, c_double_p]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)  # AttributeError here = the library does not export a declared symbol
    _fn.restype = _res
    _fn.argtypes = _args
