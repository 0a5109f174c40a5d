"""Cost and effect of the integrated log-likelihood (device_samples "loglik_int", fit_criteria(integrated=True); DESIGN.md §5f)
on one GPU, on a BASELINE config.  Prints one JSON line with the device name and power limit:
  - chain wall time with and without "loglik_int" (alternated, after a warm-up run of each);
  - gibbs_level_kernel device time per saved iteration with and without it (torch.profiler, runs of their own);
  - the criteria calls (integrated and conditional on w): wall time and fit_criteria_kernel time;
  - the store's bytes, and n_k_high and the share of k-hat > 0.5 of both criteria on the same run.

    python tools/iloo_probe.py --config C4 --keep 1000
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
    ap.add_argument("--profile-keep", type=int, default=100)
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("iloo_probe needs a GPU")
    d = synth.make_config(a.config)
    q, n = d["q"], d["y"].size
    tree = sb.make_tree(d["coords"], d["y"], d["mv_id"])
    csr = tuple(tree[k] for k in ("indexing_ptr", "indexing_idx", "parents_ptr", "parents_idx", "children_ptr", "children_idx"))
    theta = synth.theta_for(q)
    bounds, sd = synth.default_bounds(q), np.eye(theta.size) * .01
    m = sb.SpamTreeMV(d["y"], d["X"], d["coords"], d["mv_id"], tree["res_is_ref"], None, None, False, tree["block_names"],
                      tree["block_groups"], None, np.zeros(d["X"].shape[1]), theta, .1, csr=csr, keep_H=False)
    kinds = {"without": ("w",), "with": ("w", "loglik_int")}

    def run(kind, keep):
        return m.mcmc(bounds, sd, keep, 0, 1, adapting=True, rng_mode=1, seed=a.seed, device_samples=kinds[kind], save_w=False,
                      save_yhat=False)

    try:
        for kind in kinds:  # warm-up: graphs and shared-memory opt-ins of both variants
            run(kind, 5)
        t_chain = {k: [] for k in kinds}
        for _ in range(2):
            for kind in kinds:
                t0 = time.perf_counter()
                run(kind, a.keep)
                t_chain[kind].append(time.perf_counter() - t0)
        # the last run kept both stores
        crit = {"integrated": lambda: m.fit_criteria(integrated=True), "conditional": lambda: m.fit_criteria()}
        out = {}
        for key, fn in crit.items():
            first = fn()
            t_call = []
            for _ in range(3):
                t0 = time.perf_counter()
                fn()
                t_call.append(time.perf_counter() - t0)
            kh = first["pareto_k"][np.isfinite(first["lpd"])]
            out[key] = {"call_ms": [1e3 * t for t in t_call], "kernel_ms": kernel_us(fn, ("fit_criteria_kernel",)) / 1e3,
                        "n_obs": first["n_obs"], "k_threshold": first["k_threshold"], "n_k_high": first["n_k_high"],
                        "share_k_high": first["n_k_high"] / max(first["n_obs"], 1), "share_k_above_0.5": float(np.mean(kh > 0.5)),
                        "elpd_loo": first["elpd_loo_total"], "se_elpd_loo": first["se_elpd_loo"], "p_loo": first["p_loo_total"]}
        gibbs = {kind: kernel_us(lambda kind=kind: run(kind, a.profile_keep), ("gibbs_level_kernel",)) / 1e3 / a.profile_keep
                 for kind in kinds}
        line = {
            "config": a.config, "n_all": int(n), "q": q, "keep": a.keep,
            "chain_s": t_chain,
            "gibbs_ms_per_saved_iteration": gibbs, "profile_keep": a.profile_keep,
            "store_bytes": int(n) * a.keep * 8, "criteria": out,
            "device": torch.cuda.get_device_name(0), "power_limit_w": power_limit(),
        }
        print(json.dumps(line))
    finally:
        m.close()


if __name__ == "__main__":
    main()
