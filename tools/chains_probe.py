"""Cost of several chains summarised on the GPU (summarize_chains, DESIGN.md §5d) on one GPU, on a BASELINE config.  Prints
one JSON line with the device name and power limit:

- the device memory one handle takes, and what its device store of w adds, at `keep` saved iterations (from the free
  memory before and after);
- from those, the most chains of `keep` draws that fit the device at once, and the most draws per chain for `chains` chains;
- summarize_chains("w") over `chains` chains of `keep` draws next to summarize("w") over one chain: wall time of each call
  and the time of its kernel from a torch.profiler run of its own;
- the chains' wall time, and the spread of R-hat and ESS over the rows.

    python tools/chains_probe.py --config C4 --chains 4 --keep 1000
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import spamtree_b200 as sb  # noqa: E402
from spamtree_b200 import synth  # noqa: E402


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        return float(r.stdout.strip().splitlines()[0])
    except Exception:
        return None


def kernel_ms(fn, name):
    """device time (ms) of the kernels whose name contains `name`, over one profiled call of fn"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    tot = 0.0
    for e in prof.key_averages():
        if name in e.key:
            tot += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
    return tot / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C2")
    ap.add_argument("--chains", type=int, default=4)
    ap.add_argument("--keep", type=int, default=1000)
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("chains_probe needs a GPU")
    d = synth.make_config(a.config)
    q, n = d["q"], d["y"].size
    tree = sb.make_tree(d["coords"], d["y"], d["mv_id"])
    csr = tuple(tree[k] for k in ("indexing_ptr", "indexing_idx", "parents_ptr", "parents_idx", "children_ptr", "children_idx"))
    theta = synth.theta_for(q)
    bounds, sd = synth.default_bounds(q), np.eye(theta.size) * .01

    def free():
        torch.cuda.synchronize()
        return torch.cuda.mem_get_info()[0]

    free0 = free()
    total = torch.cuda.mem_get_info()[1]
    models, secs = [], []
    for k in range(a.chains):
        before = free()
        m = sb.SpamTreeMV(d["y"], d["X"], d["coords"], d["mv_id"], tree["res_is_ref"], None, None, False, tree["block_names"],
                          tree["block_groups"], None, np.zeros(d["X"].shape[1]), theta, .1, csr=csr, keep_H=False)
        m.mcmc(bounds, sd, 2, 0, 1, rng_mode=1, seed=a.seed + k, save_w=False, save_yhat=False)  # graphs and work buffers
        handle = before - free()
        t0 = time.perf_counter()
        m.mcmc(bounds, sd, a.keep, 0, 1, adapting=True, rng_mode=1, seed=a.seed + k, save_w=False, save_yhat=False,
               device_samples=("w",))
        secs.append(time.perf_counter() - t0)
        if k == 0:
            handle_bytes, store_bytes = handle, before - free() - handle
        models.append(m)
    per_draw = store_bytes / a.keep
    probs = (0.025, 0.5, 0.975)
    sb.summarize_chains(models, "w", probs)
    models[0].summarize("w", probs)
    t = time.perf_counter()
    s = sb.summarize_chains(models, "w", probs)
    t_chains = time.perf_counter() - t
    t = time.perf_counter()
    models[0].summarize("w", probs)
    t_one = time.perf_counter() - t
    k_chains = kernel_ms(lambda: sb.summarize_chains(models, "w", probs), "chains_summary_kernel")
    k_one = kernel_ms(lambda: models[0].summarize("w", probs), "summary_kernel")
    for m in models:
        m.close()
    fin = lambda v: v[np.isfinite(v)]  # noqa: E731
    line = {
        "config": a.config, "n_all": int(n), "q": q, "chains": a.chains, "keep": a.keep,
        "device_total_gb": total / 1e9, "device_free_gb_at_start": free0 / 1e9,
        "one_handle_gb": handle_bytes / 1e9, "its_w_store_gb": store_bytes / 1e9,
        "most_chains_at_keep": int(free0 // (handle_bytes + per_draw * a.keep)),
        "most_keep_at_chains": int((free0 / a.chains - handle_bytes) // per_draw),
        "chain_s": secs,
        "summarize_chains_w": {"draws_per_row": a.chains * a.keep, "call_s": t_chains, "kernel_ms": k_chains},
        "summarize_w_one_chain": {"draws_per_row": a.keep, "call_s": t_one, "kernel_ms": k_one},
        "rhat_quantiles_10_50_90_99": np.quantile(fin(s["rhat"]), (.1, .5, .9, .99)).tolist(),
        "ess_bulk_quantiles_10_50_90": np.quantile(fin(s["ess_bulk"]), (.1, .5, .9)).tolist(),
        "ess_tail_quantiles_10_50_90": np.quantile(fin(s["ess_tail"]), (.1, .5, .9)).tolist(),
        "device": torch.cuda.get_device_name(0), "power_limit_w": power_limit(),
    }
    print(json.dumps(line))


if __name__ == "__main__":
    main()
