"""Cost of the model criteria (SpamTreeMV.fit_criteria / sb.fit_criteria: PSIS-LOO, WAIC and DIC from the draws of w kept on
the device) on one GPU, on a BASELINE config.  Prints one JSON line with the device name and power limit: wall time of the
call, fit_criteria_kernel time from a torch.profiler run of its own, summarize("w") on the same store for comparison, and
the share of observed rows with k-hat above the threshold.

    python tools/fit_criteria_probe.py --config C4 --keep 1000 [--chains 4]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import spamtree_b200 as sb  # noqa: E402
from spamtree_b200 import synth  # noqa: E402
from summary_probe import kernel_us, power_limit  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C2")
    ap.add_argument("--keep", type=int, default=1000)
    ap.add_argument("--chains", type=int, default=1)
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("fit_criteria_probe needs a GPU")
    d = synth.make_config(a.config)
    q, n = d["q"], d["y"].size
    tree = sb.make_tree(d["coords"], d["y"], d["mv_id"])
    csr = tuple(tree[k] for k in ("indexing_ptr", "indexing_idx", "parents_ptr", "parents_idx", "children_ptr", "children_idx"))
    theta = synth.theta_for(q)
    bounds, sd = synth.default_bounds(q), np.eye(theta.size) * .01
    ms = []
    t_chain = []
    try:
        for k in range(a.chains):
            m = sb.SpamTreeMV(d["y"], d["X"], d["coords"], d["mv_id"], tree["res_is_ref"], None, None, False, tree["block_names"],
                              tree["block_groups"], None, np.zeros(d["X"].shape[1]), theta, .1, csr=csr, keep_H=False)
            ms.append(m)
            m.mcmc(bounds, sd, 5, 0, 1, adapting=True, rng_mode=1, seed=a.seed + k, device_samples=("w",), save_w=False,
                   save_yhat=False)  # warm-up: graphs and shared-memory opt-ins
            t0 = time.perf_counter()
            m.mcmc(bounds, sd, a.keep, 0, 1, adapting=True, rng_mode=1, seed=a.seed + k, device_samples=("w",), save_w=False,
                   save_yhat=False)
            t_chain.append(time.perf_counter() - t0)
        crit = lambda: sb.fit_criteria(ms)  # noqa: E731
        first = crit()
        t_call = []
        for _ in range(3):
            t0 = time.perf_counter()
            again = crit()
            t_call.append(time.perf_counter() - t0)
        same = all(np.array_equal(first[k], again[k], equal_nan=True) for k in first)
        k_us = kernel_us(crit, ("fit_criteria_kernel",))
        s_us = kernel_us(lambda: ms[0].summarize("w", (0.025, 0.5, 0.975)), ("summary_kernel",))
        kh = first["pareto_k"][np.isfinite(first["lpd"])]
        line = {
            "config": a.config, "n_all": int(n), "q": q, "keep": a.keep, "chains": a.chains, "draws_per_row": a.chains * a.keep,
            "chain_s": t_chain,
            "fit_criteria": {
                "call_ms": [1e3 * t for t in t_call], "kernel_ms": k_us / 1e3, "bit_identical_repeat": same,
                "bytes_read": n * a.chains * a.keep * 8,
            },
            "summarize_w_one_chain_kernel_ms": s_us / 1e3,
            "n_obs": first["n_obs"], "k_threshold": first["k_threshold"], "n_k_high": first["n_k_high"],
            "share_k_high": first["n_k_high"] / max(first["n_obs"], 1),
            "share_k_above_0.5": float(np.mean(kh > 0.5)), "share_k_inf": float(np.mean(np.isinf(kh))),
            "elpd_loo": first["elpd_loo_total"], "se_elpd_loo": first["se_elpd_loo"], "p_loo": first["p_loo_total"],
            "elpd_waic": first["elpd_waic_total"], "p_waic": first["p_waic_total"], "dic": first["dic"], "p_dic": first["p_dic"],
            "device": torch.cuda.get_device_name(0), "power_limit_w": power_limit(),
        }
        print(json.dumps(line))
    finally:
        for m in ms:
            m.close()


if __name__ == "__main__":
    main()
