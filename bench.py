#!/usr/bin/env python
"""bench.py — MCMC iterations/s of the SpamTrees hot path on N B200s (BASELINE.json metric), one process per GPU.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N ...            # the reference algorithm on the host cores (CPU oracle): --steps full
                                                           # CPU iterations, about 1.3 s each at C4 on 16 cores
  python bench.py --steps K --dump-outputs DIR             # + the last timed step's outputs as DIR/<name>.npy

A "step" is one MCMC iteration of the hot path (spamtree_fit.cpp:167-330 minus predict/save): GIBBS sweep over w + LLW +
BUILD at a proposed theta + accept/swap + tausq + beta.  The workload is BASELINE config C4 (q=3, n=1M) at every N: at
N>1 the ONE problem is cut into subtrees (spamtree_b200/partition.py), one rank per GPU, NCCL carrying the log-density
scalars, the cut-level messages and the beta/tausq statistics ("strong" scaling; DESIGN.md §7).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "mcmc_iterations_per_sec"
UNIT = "it/s"


def build_dram_traffic(workload):
    """DRAM bytes of the build_level_kernel launches of ONE BUILD from the tracked ncu summary (profiles/*_build_dram.json,
    written by tools/ncu_build_dram.py) — only while the kernel sources it was measured on are the ones that run now"""
    import glob
    import hashlib
    h = hashlib.sha1()
    for f in ["spamtree_b200/csrc/st_build.cu", "spamtree_b200/csrc/st_device.cuh", "spamtree_b200/csrc/st_build_plan.cuh"]:
        h.update(open(os.path.join(ROOT, f), "rb").read())
    sha = h.hexdigest()
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_build_dram.json")), reverse=True):
        d = json.load(open(path))
        if d.get("workload") == workload and d.get("sources_sha1") == sha:
            return d["dram_bytes"], f"{os.path.relpath(path, ROOT)} (ncu dram__bytes_read.sum + dram__bytes_write.sum over the build_level_kernel launches of one BUILD; kernel sources {sha[:10]})"
    return None, f"no ncu summary under profiles/ matches the kernel sources that ran ({sha[:10]}): not reported"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "MEASURED_PEAKS.json"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """samples nvidia-smi clocks / throttle reasons during the timed region"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, False, []

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        try:
            self.proc.terminate()
        except Exception:
            pass
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def build_problem(workload, seed):
    import spamtree_b200 as sb
    from spamtree_b200 import synth
    d = synth.make_config(workload, seed=seed)
    t = sb.make_tree(d["coords"], d["y"], d["mv_id"])
    csr = (t["indexing_ptr"], t["indexing_idx"], t["parents_ptr"], t["parents_idx"], t["children_ptr"], t["children_idx"])
    return d, t, csr, synth.theta_for(d["q"])


def proposals(theta, k, seed):
    """a fixed sequence of small random-walk proposals around the parity-point theta (same for every arm)"""
    rng = np.random.default_rng(seed)
    return [theta * (1 + 0.002 * rng.standard_normal(theta.size)) for _ in range(k)]


DUMP_ROWS = 1 << 21  # rows of w and XB written by --dump-outputs: 2 x 16 MB of float64 at most


def dump_outputs(path, gm, last):
    """what the last timed step computed, as a caller of bench_iteration receives it: its return values (log-density of the
    proposal, of the previous current state, 1 if the proposal's BUILD was acceptable) and the state it leaves (w, beta,
    1 / tausq, X beta).  Above DUMP_ROWS rows, w and XB are kept at a fixed, seeded sample of rows, written as rows.npy."""
    os.makedirs(path, exist_ok=True)
    pr = gm.params()
    out = {"loglik": last, "w": gm.w, "beta": pr["Bcoeff"], "tausq_inv": pr["tausq_inv"], "xb": pr["XB"]}
    if gm.n_all > DUMP_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(gm.n_all, DUMP_ROWS, replace=False))
        out.update(w=out["w"][rows], xb=out["xb"][rows], rows=rows)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def measure_fp64_peak(torch, dev):
    """cuBLAS DGEMM 4096^3 back to back: the FP64 roofline denominator (MEASURED_PEAKS.json carries no FP64 figure)"""
    n = 4096
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    torch.cuda.synchronize(dev)
    best = 0.0
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(4):
            torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize(dev)
        best = max(best, 4 * 2 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    del a, b
    return best


def host_threads():
    """the cores this process may run on (torchrun exports OMP_NUM_THREADS=1, which must not throttle the CPU arm)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_backend():
    """dense kernels of the CPU arm: scipy's bundled OpenBLAS when it is there (the reference reaches BLAS/LAPACK through
    Armadillo, SURVEY §8c), else the port's own loops.  The parity tests always use the loops."""
    from oracle import oracle as orc
    path = orc.use_blas(True)
    return ("port+blas: dense kernels by " + os.path.basename(path) + " (1 thread per call), OpenMP over the blocks of a level") if path else \
        "port: plain loops, OpenMP over the blocks of a level"


def cpu_baseline_sample(workload, d, t, csr, theta, iters=1, blas=True):
    """the oracle (restated reference algorithm, OpenMP over the blocks of a level like spamtree_model.cpp:850) timed on
    the host cores on the SAME workload: one untimed BUILD to initialise, then `iters` timed iterations"""
    from oracle import oracle as orc
    backend = cpu_backend() if blas else (orc.use_blas(False) or "port: plain loops, OpenMP over the blocks of a level")
    om = orc.OracleModel(d["y"], d["X"], d["coords"], d["mv_id"], t["res_is_ref"], csr, False, t["block_names"], t["block_groups"],
                         np.zeros(3), theta, 0.1, flags=orc.FLAG_LEAN)
    orc.lib().or_set_threads(host_threads())
    cores = orc.lib().or_max_threads()
    om.get_loglik_comps_w(0)
    props = proposals(theta, iters + 1, 99)
    om.timed_iteration(props[iters], False)  # warm-up: first touch of the per-block state
    ts = [om.timed_iteration(props[i], do_swap=(i % 4 == 3)) for i in range(iters)]
    om.close()
    orc.use_blas(False)
    return {"value": 1.0 / float(np.mean(ts)), "unit": UNIT, "cores": int(cores), "kind": "port", "backend": backend,
            "sample": f"{workload} full tree, lean-state oracle (identical arithmetic per block, P x P scratch not kept): "
                      f"1 untimed BUILD + 1 untimed iteration, then {iters} timed iteration(s) of {float(np.mean(ts)):.2f} s"}, ts


def config_of(workload, d, t, n_gpus, gc=None):
    """the `config` object BOTH arms print, value for value: the workload and how the job of N GPUs divides it (the CPU arm
    times the same workload on the host cores; what it ran on is in its `cpu_baseline`)"""
    if n_gpus > 1 and gc is None:
        from spamtree_b200 import partition as part
        gc = part.plan(t, d["y"], n_gpus)["gc"]
    par = "single GPU" if n_gpus == 1 else (f"{n_gpus} ranks, subtree partition below tree level {gc} (levels above replicated); NCCL all-reduce of "
                                            "3 log-density scalars (x2), cut-level messages and beta/tausq statistics per iteration")
    return {"workload": workload, "n": int(d["y"].size), "q": int(d["q"]), "p": 3, "blocks": int(t["n_blocks"]),
            "levels": int(len(t["res_is_ref"])), "theta": "fixed parity point, 0.2% random-walk proposals, every 4th accepted",
            "l2": "working set (G, Ri of both theta slots, >3 GB at C4) is larger than the 126 MB L2; no flush needed",
            "parallelism": par}


def run_reference(args, rank, world, emit):
    if rank != 0:
        return
    d, t, csr, theta = build_problem(args.workload, 2021)
    warm = max(args.warmup, 3)  # the same warm-up policy as the product arm
    from oracle import oracle as orc
    om = orc.OracleModel(d["y"], d["X"], d["coords"], d["mv_id"], t["res_is_ref"], csr, False, t["block_names"], t["block_groups"],
                         np.zeros(3), theta, 0.1, flags=orc.FLAG_LEAN)
    orc.lib().or_set_threads(host_threads())  # every host thread, also under torchrun (which exports OMP_NUM_THREADS=1)
    cores = orc.lib().or_max_threads()
    om.get_loglik_comps_w(0)
    props = proposals(theta, warm + args.steps, 99)
    # the faster backend of the port for this workload (host OpenBLAS pays off on the big trees, the plain loops on the small
    # ones): one probe iteration each, then the warm-up and the timed iterations with the winner
    backend = "port: plain loops, OpenMP over the blocks of a level"
    if not args.cpu_loops:
        om.timed_iteration(props[0], False)
        t_loops = om.timed_iteration(props[0], False)
        b = cpu_backend()
        om.timed_iteration(props[0], False)
        t_blas = om.timed_iteration(props[0], False)
        if b.startswith("port+blas") and t_blas < t_loops:
            backend = b
        else:
            orc.use_blas(False)
    for i in range(warm):
        om.timed_iteration(props[i], do_swap=(i % 4 == 3))
    steps = min(args.steps, args.ref_steps) if args.ref_steps > 0 else args.steps
    ts = [om.timed_iteration(props[warm + i], do_swap=(i % 4 == 3)) for i in range(steps)]
    v = steps / float(np.sum(ts))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": 1e3 / v, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_of(args.workload, d, t, args.gpus),
            "note": "CPU arm: the reference algorithm (oracle port, OpenMP over the blocks of a level) on the host cores; --steps iterations, "
                    "fewer only where --ref-steps caps them",
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": int(cores), "kind": "port", "backend": backend,
                             "sample": f"{steps} timed iteration(s) after {warm} warm-up on the full {args.workload} tree, lean-state oracle"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed iterations, in both arms; with --impl reference each is a full CPU iteration (about 1.3 s at C4 on 16 "
                         "host cores), so the run takes about that many times longer (--ref-steps caps them)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C4", choices=["C1", "C2", "C3", "C4", "C5"])
    ap.add_argument("--ref-steps", type=int, default=0, help="cap on the timed iterations of --impl reference (0: --steps)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-loops", action="store_true", help="CPU arm with the port's own loops instead of the host's OpenBLAS")
    ap.add_argument("--no-predict-leg", action="store_true", help="skip the extra end-to-end leg with prediction on a thin schedule")
    ap.add_argument("--e2e-steps", type=int, default=0, help="iterations of the end-to-end leg (default: --steps)")
    ap.add_argument("--e2e-sd", type=float, default=1e-8,
                    help="diagonal of mcmcsd in the end-to-end leg (the proposal covariance in logit space, spamtree_fit.cpp:95): small "
                         "enough that a share of the proposals is accepted at n = 1M, as in a tuned chain; the accepted count is reported")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64), to compare builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # stdout carries exactly ONE JSON line: anything a library prints there (NCCL's version banner ...) goes to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        os.write(real_stdout, (json.dumps(line) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.impl == "reference" or world > 1):
        ap.error("--dump-outputs writes the outputs of the CUDA path on one GPU")
    if args.impl == "reference":
        run_reference(args, rank, world, emit)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import spamtree_b200 as sb
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # one problem; at N > 1 every rank builds the same tree and keeps its subtrees plus the replicated top levels
    d, t, csr, theta = build_problem(args.workload, 2021)
    if world > 1:
        from spamtree_b200 import dist as sdist
        gm, sp, pl = sdist.partitioned_model(d, t, theta, np.zeros(3), 0.1, rank, world, local_rank, sdist.make_allreduce(dev))
    else:
        sp, pl = None, None
        gm = sb.SpamTreeMV(d["y"], d["X"], d["coords"], d["mv_id"], t["res_is_ref"], None, None, False, t["block_names"], t["block_groups"],
                           None, np.zeros(3), theta, 0.1, csr=csr, keep_H=False, device=local_rank)
    gm.set_beta_index(False)  # the corrected row index at every N (a partition supports no other): same chain for every N
    gm.get_loglik_comps_w(0)
    gm.get_loglik_comps_w(1)
    props = proposals(theta, args.warmup + args.steps, 99)
    for i in range(args.warmup):
        gm.bench_iteration(props[i], do_swap=(i % 4 == 3), seed=i)
    probe_ll, probe_ld = gm.get_loglik_w(0)
    fp64_peak = measure_fp64_peak(torch, dev) if rank == 0 else 0.0

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    c0 = gm.counters()
    phase = np.zeros(6)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        last, ms = gm.bench_iteration(props[args.warmup + i], do_swap=(i % 4 == 3), seed=1000 + i)
        phase += ms
    gm.sync()
    barrier()
    elapsed = time.perf_counter() - t0
    c1 = gm.counters()
    clocks = sampler.finish() if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, gm, last)
    # device time of the step: CUDA events around the whole iteration on the launching stream (the per-phase times do not
    # add up to it: the upper levels of BUILD run on a second stream underneath the Gibbs sweep)
    dev_ms = float(phase[4])
    tt = torch.tensor([elapsed, dev_ms * 1e-3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    elapsed_max, dev_s_max = float(tt[0]), float(tt[1])
    value = args.steps / elapsed_max  # one chain: iterations of the whole job per second

    # end-to-end leg: the public driver (spamtree_mv_mcmc loop) with host buffers; every iteration is a saved one
    # (theta', tausq, beta go host->device; the 3 log-density scalars, the sufficient statistics and w come back)
    e2e_steps = args.e2e_steps or args.steps
    from spamtree_b200 import synth
    bounds = synth.default_bounds(d["q"])
    npar = theta.size
    # warm-up of the end-to-end leg, outside its timed region (like the --warmup steps of the device-timed leg): first use of
    # the public driver on this handle (CUDA-graph instantiation, first NCCL call per buffer, page-locking of the outputs)
    gm.mcmc(bounds, np.eye(npar) * args.e2e_sd, keep=max(args.warmup, 3), burn=0, thin=1, adapting=True, rng_mode=1, seed=4,
            sample_predicts=False, save_w=True, save_yhat=False, faithful_beta_index=(world == 1))
    barrier()
    res = gm.mcmc(bounds, np.eye(npar) * args.e2e_sd, keep=e2e_steps, burn=0, thin=1, adapting=True, rng_mode=1, seed=5,
                  sample_predicts=False, save_w=True, save_yhat=False, faithful_beta_index=(world == 1))
    te = torch.tensor([res["mcmc_time"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = e2e_steps / float(te[0])
    # the same driver with prediction at the missing rows (predict_std, spamtree_model.cpp:1234-1358) on a thin schedule,
    # as SURVEY §8d asks: every 5th iteration is a saved one (predict + w to the host).  Single GPU only, reported beside e2e.
    e2e_pred = None
    if world == 1 and not args.no_predict_leg:
        try:
            thin, kp = 5, max(2, e2e_steps // 5)
            rp = gm.mcmc(bounds, np.eye(npar) * args.e2e_sd, keep=kp, burn=0, thin=thin, adapting=True, rng_mode=1, seed=6,
                         sample_predicts=True, save_w=True, save_yhat=False, faithful_beta_index=True)
            e2e_pred = {"value": kp * thin / float(rp["mcmc_time"]), "unit": UNIT, "iterations": kp * thin, "thin": thin,
                        "accepted": int(rp["n_accepted"]),
                        "note": "sample_predicts = TRUE: prediction blocks rebuilt and sampled, w saved, on every 5th iteration"}
        except Exception as ex:  # a reported extra, never allowed to take the bench line down
            e2e_pred = {"value": None, "unit": UNIT, "error": str(ex)[:200]}
    cnt = gm.counters()
    tw = torch.tensor([cnt["f_alg"], cnt["f_exec"], c1["launches"] - c0["launches"], cnt["f_alg_build"], cnt["f_exec_build"],
                       cnt["b_alg_build"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tw)  # work and launches of the whole job (replicated top levels counted on every rank)
    # BUILD time of the job: max over ranks of the per-rank mean.  Where the upper levels run on the second stream (small trees,
    # ranks of a partition) their elapsed time there is added: pessimistic, it includes their waiting behind the sweep
    tb = torch.tensor([float(phase[2] + phase[5]) / args.steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tb, op=dist.ReduceOp.MAX)
    n_all, q, p = int(d["y"].size), int(d["q"]), 3
    n_local = n_all if sp is None else int(sp["y"].size)
    # per rank and iteration: the device-resident chain sends nothing per iteration (its state goes up once per run) and
    # brings back the saved w plus the saved theta / beta / tausq; the chain state comes back once per run
    chain_bytes = int(cnt["chain_state_bytes"])
    h2d = int(np.ceil(chain_bytes / e2e_steps))
    d2h = 8 * (n_local + npar + q + p * q) + int(np.ceil(chain_bytes / e2e_steps))

    if rank == 0:
        hbm_peak, peak_src = load_peaks()
        build_ms = float(tb[0])
        f_alg, f_exec, f_alg_build, f_exec_build, b_alg_build = (float(tw[i]) for i in (0, 1, 3, 4, 5))
        fp64_peak_job = fp64_peak * world
        traffic, traffic_note = build_dram_traffic(args.workload) if world == 1 else (None, "single-GPU figure only")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * elapsed_max / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": config_of(args.workload, d, t, world, pl["gc"] if pl else None),
            # log-density of the current slot after the warm-up iterations (fixed proposals, fixed accept pattern, random
            # numbers keyed by the row's id in the whole problem): the same number at every N up to summation order
            "parity_probe": {"after_warmup_iterations": args.warmup, "loglik_w": probe_ll, "logdetCi": probe_ld},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps, "accepted": int(res["n_accepted"]), "chol_fail": int(res["n_chol_fail"]), "mcmcsd_diag": args.e2e_sd,
                    "path": "SpamTreeMV.mcmc -> st_mcmc_run (spamtree_mv_mcmc loop, device-resident chain), host output buffers, every "
                            "iteration saved (w, theta, beta, tausq copied to the host); warm-up run outside the timed region"},
            "e2e_with_predict": e2e_pred,
            "gpu_launches": int(tw[2]),
            "device_ms_per_step": {"gibbs": float(phase[0]) / args.steps, "llw": float(phase[1]) / args.steps,
                                   "build": build_ms, "beta_tausq": float(phase[3]) / args.steps, "max_over_ranks_total": 1e3 * dev_s_max / args.steps,
                                   "build_upper_levels_overlapped": float(phase[5]) / args.steps,
                                   "note": "rank 0's CUDA-event phase times; build = main-stream BUILD (+ accept, + the deferred half of an accepted "
                                           "proposal) + the upper levels' elapsed time on the second stream where they overlap the sweep"},
            # dominant kernel: build_level_kernel (all level launches of one BUILD, ~80 % of the step).  achieved = F_build
            # (SURVEY §8d formula summed over the actual tree) / the BUILD time measured here with CUDA events on the
            # launching stream; peak = cuBLAS DGEMM measured in this run (MEASURED_PEAKS.json has no FP64 figure)
            "roofline": {"bound": "tensor", "pipe": "FP64 tensor-core MMA (mma.sync m8n8k4 f64; tcgen05 has no FP64 kind) + FP64 FMA pipe for the covariance kernels",
                         "kernel": "build_level_kernel (all level launches of one BUILD)",
                         "achieved": f_alg_build / (build_ms * 1e-3) / 1e12 if build_ms > 0 else None,
                         "peak": fp64_peak_job, "unit": "TFLOP/s", "frac": None,
                         "traffic": traffic,
                         "traffic_note": traffic_note,
                         "achieved_executed": f_exec_build / (build_ms * 1e-3) / 1e12 if build_ms > 0 else None,
                         "algorithmic_output_bytes": b_alg_build,
                         "whole_step": {"achieved": None, "achieved_executed": None, "frac": None},
                         "peak_source": "cuBLAS DGEMM 4096^3 measured in this run (MEASURED_PEAKS.json has no FP64 figure); HBM peak " + peak_src,
                         "f_alg_per_iteration": f_alg, "f_executed_per_iteration": f_exec,
                         "f_alg_build": f_alg_build, "f_executed_build": f_exec_build, "hbm_peak_gbs": hbm_peak},
        }
        step_s = elapsed_max / args.steps
        rf = line["roofline"]
        if fp64_peak and rf["achieved"] is not None:
            rf["frac"] = rf["achieved"] / fp64_peak_job
            rf["frac_executed"] = rf["achieved_executed"] / fp64_peak_job
        rf["whole_step"] = {"achieved": f_alg / step_s / 1e12, "achieved_executed": f_exec / step_s / 1e12,
                            "frac": (f_alg / step_s / 1e12) / fp64_peak_job if fp64_peak else None}
        if world == 1 and not args.no_cpu_baseline:
            try:
                # both backends of the port (host OpenBLAS / plain loops); the FASTER one is the baseline, the other is shown
                cands = [cpu_baseline_sample(args.workload, d, t, csr, theta, iters=3, blas=b)[0] for b in ((False,) if args.cpu_loops else (True, False))]
                cands.sort(key=lambda c: -c["value"])
                line["cpu_baseline"] = cands[0]
                if len(cands) > 1:
                    line["cpu_baseline_other_backend"] = cands[1]
            except Exception as ex:  # the baseline is reported, never required for the GPU number
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": None, "kind": "port", "sample": f"failed: {ex}"}
        emit(line)
    gm.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
