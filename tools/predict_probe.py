"""Cost of prediction at new locations (SpamTreeMV.predict_new) on one GPU: a short device-resident chain on a BASELINE
config, then draws at a regular raster of new points from its saved samples — once at the chain's own thetas (a BUILD per
change of theta) and once with a theta of its own per sample (a BUILD every sample).  Prints one JSON line: per pass, ms per
sample (end to end, and split by kernel into the reference-level BUILD, the prediction pass and the copies, from a
torch.profiler run of its own), the BUILDs run and rows x samples per second; and the device name and power limit the
numbers were taken on.

    python tools/predict_probe.py --config C4 --raster 1000 --samples 64
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C2")
    ap.add_argument("--raster", type=int, default=1000, help="new points: raster x raster over the unit square")
    ap.add_argument("--samples", type=int, default=64)
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("predict_probe needs a GPU")
    d = synth.make_config(a.config)
    q = d["q"]
    g = (np.arange(a.raster) + .5) / a.raster
    cn = np.stack(np.meshgrid(g, g, indexing="ij"), -1).reshape(-1, 2)
    nn = cn.shape[0]
    mvn = 1 + np.arange(nn) % q
    xn = np.random.default_rng(a.seed).standard_normal((nn, d["X"].shape[1]))
    t0 = time.perf_counter()
    tree = sb.make_tree(d["coords"], d["y"], d["mv_id"], coords_new=cn, mv_id_new=mvn)
    t_tree = time.perf_counter() - t0
    csr = tuple(tree[k] for k in ("indexing_ptr", "indexing_idx", "parents_ptr", "parents_idx", "children_ptr", "children_idx"))
    theta = synth.theta_for(q)
    m = sb.SpamTreeMV(d["y"], d["X"], d["coords"], d["mv_id"], tree["res_is_ref"], None, None, False, tree["block_names"],
                      tree["block_groups"], None, np.zeros(d["X"].shape[1]), theta, .1, csr=csr, keep_H=False)
    S = a.samples
    bounds = synth.default_bounds(q)
    res = m.mcmc(bounds, np.eye(theta.size) * .01, S, 0, 1, adapting=True, rng_mode=1, seed=a.seed, save_yhat=False)
    n_theta_changes = 1 + int(np.sum(np.any(res["theta_mcmc"][:, 1:] != res["theta_mcmc"][:, :-1], axis=0)))
    # warm-up of every launch shape, then per pass: the end-to-end timing (the call synchronises once, at its end) and the
    # kernel split in a profiled call of its own
    m.predict_new(cn, xn, mvn, tree["new"], {k: (v[:, :2] if k != "beta_mcmc" else v[:, :2, :]) for k, v in res.items()
                                             if k in ("theta_mcmc", "tausq_mcmc", "w_mcmc", "beta_mcmc")})
    from torch.profiler import ProfilerActivity, profile

    def measure(samples):
        t0 = time.perf_counter()
        out = m.predict_new(cn, xn, mvn, tree["new"], samples, seed=a.seed)
        t_call = time.perf_counter() - t0
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            m.predict_new(cn, xn, mvn, tree["new"], samples, seed=a.seed)
        split = {"ref_build": 0.0, "predict_pass": 0.0, "copies": 0.0, "other": 0.0}
        for e in prof.key_averages():
            us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            name = e.key
            if "build_level_kernel_ref" in name:
                split["ref_build"] += us
            elif any(k in name for k in ("build_level_kernel<3>", "predict_draw_kernel", "gather_sample_kernel", "predict_moments")):
                split["predict_pass"] += us
            elif "memcpy" in name.lower():
                split["copies"] += us
            elif name.startswith("Memset") or "kernel" in name.lower():
                split["other"] += us
        return {
            "n_builds": out["n_builds"],
            "ms_per_sample": 1e3 * t_call / S,
            "ms_per_sample_kernels": {k: v / 1e3 / S for k, v in split.items()},
            "build_share_of_kernel_time": split["ref_build"] / max(sum(split.values()), 1e-30),
            "rows_x_samples_per_s": nn * S / t_call,
        }

    chain = measure(res)
    # every sample at a theta of its own (the chain's first, scaled by 1 + 1e-9 (s + 1)): one reference BUILD per sample
    th_all = res["theta_mcmc"][:, :1] * (1.0 + 1e-9 * np.arange(1, S + 1))[None, :]
    every = measure(dict(res, theta_mcmc=th_all))
    m.close()
    line = {
        "config": a.config, "n_all": int(d["y"].size), "q": q, "n_new": nn, "samples": S,
        "theta_changes_in_chain": n_theta_changes,
        "chain_samples": chain, "theta_changes_every_sample": every,
        "tree_attach_s_incl_tree": t_tree,
        "device": torch.cuda.get_device_name(0), "power_limit_w": power_limit(),
    }
    print(json.dumps(line))


if __name__ == "__main__":
    main()
