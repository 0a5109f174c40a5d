"""Cost of keeping draws on the device and summarising them there (SpamTreeMV.mcmc(device_samples=...), summarize,
predict_new(samples=None)) on one GPU, on a BASELINE config.  Prints one JSON line with the device name and power limit:

- end-to-end it/s of a device-resident run of `keep` saved iterations that copies w and yhat to host arrays, and of the same
  run with the device store and no host arrays (same seed: the same chain);
- summarize("w") with three probs: wall time of the call, summary_kernel time from a torch.profiler run of its own, and the
  bytes the kernel reads (n_all x keep x 8) over the kernel time, against the 6.5 TB/s HBM copy bandwidth;
- per-sample predict_new on a raster x raster grid from `samples` saved iterations: from host arrays, from the store with
  the draws copied out, and from the store with the draws kept on the device.

    python tools/summary_probe.py --config C4 --keep 1000 --raster 1000 --samples 64
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

HBM_COPY_TBS = 6.5  # device-to-device copy bandwidth of one B200 the project measures against (DESIGN.md §4)


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        return float(r.stdout.strip().splitlines()[0])
    except Exception:
        return None


def kernel_us(fn, names):
    """device time (us) of the kernels whose name contains one of `names`, over one profiled call of fn"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    tot = 0.0
    for e in prof.key_averages():
        if any(n in e.key for n in names):
            tot += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
    return tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C2")
    ap.add_argument("--keep", type=int, default=1000)
    ap.add_argument("--raster", type=int, default=1000)
    ap.add_argument("--samples", type=int, default=64)
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("summary_probe needs a GPU")
    d = synth.make_config(a.config)
    q, n = d["q"], d["y"].size
    g = (np.arange(a.raster) + .5) / a.raster
    cn = np.stack(np.meshgrid(g, g, indexing="ij"), -1).reshape(-1, 2)
    nn = cn.shape[0]
    mvn = 1 + np.arange(nn) % q
    xn = np.random.default_rng(a.seed).standard_normal((nn, d["X"].shape[1]))
    tree = sb.make_tree(d["coords"], d["y"], d["mv_id"], coords_new=cn, mv_id_new=mvn)
    csr = tuple(tree[k] for k in ("indexing_ptr", "indexing_idx", "parents_ptr", "parents_idx", "children_ptr", "children_idx"))
    theta = synth.theta_for(q)
    m = sb.SpamTreeMV(d["y"], d["X"], d["coords"], d["mv_id"], tree["res_is_ref"], None, None, False, tree["block_names"],
                      tree["block_groups"], None, np.zeros(d["X"].shape[1]), theta, .1, csr=csr, keep_H=False)
    bounds, sd = synth.default_bounds(q), np.eye(theta.size) * .01

    def run(keep, **kw):
        t0 = time.perf_counter()
        r = m.mcmc(bounds, sd, keep, 0, 1, adapting=True, rng_mode=1, seed=a.seed, **kw)
        return r, time.perf_counter() - t0

    run(5, device_samples=("w", "yhat"))  # warm-up: graphs, shared-memory opt-ins, the copy stream
    run(5)
    host_gb = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES") / 2 ** 30
    # the store run first (no host arrays), then the same chain into host arrays (2 x n x keep doubles on the host)
    rs, ts = run(a.keep, device_samples=("w", "yhat"), save_w=False, save_yhat=False)
    probs = (0.025, 0.5, 0.975)
    m.summarize("w", probs)
    t_sum = []
    for _ in range(3):
        t0 = time.perf_counter()
        m.summarize("w", probs)
        t_sum.append(time.perf_counter() - t0)
    k_us = kernel_us(lambda: m.summarize("w", probs), ("summary_kernel",))
    bytes_read = n * a.keep * 8
    m.mcmc(bounds, sd, 1, 0, 1, rng_mode=1, device_samples=())  # frees the store before the host-array run
    rh, th = run(a.keep)
    same_chain = bool(np.array_equal(rh["theta_mcmc"], rs["theta_mcmc"]))
    mt_host, mt_store = rh["mcmc_time"], rs["mcmc_time"]
    del rh
    # prediction: `samples` saved iterations, w kept on the device and in host arrays
    S = a.samples
    rp, _ = run(S, device_samples=("w",), save_yhat=False)
    new = tree["new"]
    m.predict_new(cn, xn, mvn, new, rp, seed=a.seed)  # warm-up of every launch shape
    m.predict_new(cn, xn, mvn, new, None, seed=a.seed)

    def timed(fn):
        t0 = time.perf_counter()
        out = fn()
        return out, time.perf_counter() - t0

    ph, t_ph = timed(lambda: m.predict_new(cn, xn, mvn, new, rp, seed=a.seed))
    pd, t_pd = timed(lambda: m.predict_new(cn, xn, mvn, new, None, seed=a.seed))
    pk, t_pk = timed(lambda: m.predict_new(cn, xn, mvn, new, None, seed=a.seed, draws=False, keep_draws=True))
    same_pred = bool(np.array_equal(ph["w_new"], pd["w_new"]) and np.array_equal(ph["w_new_mean"], pk["w_new_mean"]))
    t_sn = timed(lambda: m.summarize("yhat_new", probs))[1]
    m.close()
    line = {
        "config": a.config, "n_all": int(n), "q": q, "keep": a.keep, "host_memory_gb": round(host_gb, 1),
        "chain_host_arrays": {"s": th, "it_per_s": a.keep / th, "mcmc_time_s": mt_host},
        "chain_device_store": {"s": ts, "it_per_s": a.keep / ts, "mcmc_time_s": mt_store},
        "same_chain": same_chain,
        "summarize_w_3probs": {
            "call_ms": [1e3 * t for t in t_sum], "kernel_ms": k_us / 1e3, "bytes_read": bytes_read,
            "tb_per_s": bytes_read / (k_us * 1e-6) / 1e12 if k_us else None,
            "share_of_hbm_copy_bw": bytes_read / (k_us * 1e-6) / (HBM_COPY_TBS * 1e12) if k_us else None,
        },
        "predict_new": {
            "n_new": nn, "samples": S, "n_builds": ph["n_builds"], "same_outputs": same_pred,
            "ms_per_sample_host_arrays": 1e3 * t_ph / S, "ms_per_sample_store_draws_to_host": 1e3 * t_pd / S,
            "ms_per_sample_store_draws_on_device": 1e3 * t_pk / S, "summarize_yhat_new_ms": 1e3 * t_sn,
        },
        "device": torch.cuda.get_device_name(0), "power_limit_w": power_limit(),
    }
    print(json.dumps(line))


if __name__ == "__main__":
    main()
