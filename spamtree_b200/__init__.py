"""spamtree_b200 — B200-native implementation of the SpamTrees per-iteration MCMC hot path (see DESIGN.md)."""
from .api import (CrossCovarianceAG10, SpamTreeError, SpamTreeMV, kthresholds, limited_edges_csr, make_edges,  # noqa: F401
                  make_edges_limited, make_tree, number_revalue, part_axis_parallel_lmt, spamtree, spamtree_mv_mcmc,
                  summarize_chains, summarize_draws, fit_criteria, fit_criteria_loglik, loo_compare,
                  par_huvtransf_fwd, par_huvtransf_back, mh_propose, do_I_accept, ram_adapt)

__all__ = ["spamtree", "CrossCovarianceAG10", "spamtree_mv_mcmc", "SpamTreeMV", "make_tree", "make_edges",
           "make_edges_limited", "par_huvtransf_fwd", "par_huvtransf_back", "kthresholds", "part_axis_parallel_lmt", "number_revalue", "SpamTreeError",
           "summarize_chains", "summarize_draws", "fit_criteria", "fit_criteria_loglik", "loo_compare"]
