"""bench.py's CPU-runnable arm (--impl reference: the reference algorithm's CPU port on the host cores) prints ONE JSON line
with the keys the measurement contract names; the CUDA arm needs a GPU and is exercised by the driver."""
import json

import numpy as np
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra, env=None):
    e = dict(os.environ)
    e.update(env or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "C1", "--steps", "3",
                        "--warmup", "1", *extra], capture_output=True, text=True, cwd=ROOT, env=e, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return [l for l in r.stdout.splitlines() if l.strip()]


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "mcmc_iterations_per_sec" and d["unit"] == "it/s"
    # (both arms raise --warmup to at least 3 and report what they ran)
    assert d["steps"] == 3 and d["warmup"] == 3 and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["value"] > 0 and abs(d["ms_per_step"] * d["value"] - 1e3) < 1e-6 * 1e3
    assert d["vs_baseline"] is None and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["config"]["workload"] == "C1" and d["config"]["n"] == 625
    assert set(d["config"]) == {"workload", "n", "q", "p", "blocks", "levels", "theta", "l2", "parallelism"}  # = the product arm's keys
    cb, e2e = d["cpu_baseline"], d["e2e"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert e2e == {"value": d["value"], "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_runs_on_rank_0_only():
    # under torchrun the other ranks exit 0 without work (and without output)
    lines = _run("--gpus", "2", env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert lines == []


import pytest  # noqa: E402


def test_dump_outputs_writes_float64_and_samples_large_outputs(tmp_path, monkeypatch):
    """--dump-outputs: every array as float64; above DUMP_ROWS rows, w and XB at a fixed sample of rows (the same every run)"""
    sys.path.insert(0, ROOT)
    import bench

    class Model:
        n_all = 50
        w = np.arange(50.0)

        def params(self):
            return {"Bcoeff": np.ones((3, 2)), "tausq_inv": np.ones(2, dtype=np.float32), "XB": -np.arange(50.0)}

    monkeypatch.setattr(bench, "DUMP_ROWS", 20)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), Model(), np.array([-1.5, -2.5, 1.0]))
    got = {f.stem: np.load(f) for f in sorted((tmp_path / "a").glob("*.npy"))}
    assert set(got) == {"loglik", "w", "beta", "tausq_inv", "xb", "rows"} and all(a.dtype == np.float64 for a in got.values())
    rows = got["rows"].astype(int)
    assert rows.size == 20 and np.all(np.diff(rows) > 0)
    assert np.array_equal(got["w"], rows) and np.array_equal(got["xb"], -rows)
    assert all(np.array_equal(np.load(tmp_path / "b" / f"{k}.npy"), v) for k, v in got.items())


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr and not any(tmp_path.iterdir())


@pytest.mark.gpu
def test_product_arm_dumps_the_last_steps_outputs(tmp_path):
    """--dump-outputs holds what the LAST timed step returned and left: bench.py's step sequence on C1 (same problem, same
    proposals and seeds) replayed in this process must give every file exactly; --steps sets the timed steps"""
    warmup, steps = 3, 5
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "C1", "--steps", str(steps), "--warmup", str(warmup),
                        "--no-cpu-baseline", "--no-predict-leg", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == steps
    got = {f.stem: np.load(f) for f in sorted(tmp_path.glob("*.npy"))}
    assert set(got) == {"loglik", "w", "beta", "tausq_inv", "xb"} and all(v.dtype == np.float64 for v in got.values())
    sys.path.insert(0, ROOT)
    import bench
    import spamtree_b200 as sb
    d, t, csr, theta = bench.build_problem("C1", 2021)
    gm = sb.SpamTreeMV(d["y"], d["X"], d["coords"], d["mv_id"], t["res_is_ref"], None, None, False, t["block_names"], t["block_groups"],
                       None, np.zeros(3), theta, 0.1, csr=csr, keep_H=False, device=0)
    gm.set_beta_index(False)
    gm.get_loglik_comps_w(0)
    gm.get_loglik_comps_w(1)
    props = bench.proposals(theta, warmup + steps, 99)
    for i in range(warmup):
        gm.bench_iteration(props[i], do_swap=(i % 4 == 3), seed=i)
    gm.get_loglik_w(0)  # bench.py's parity probe
    outs = [gm.bench_iteration(props[warmup + i], do_swap=(i % 4 == 3), seed=1000 + i)[0] for i in range(steps)]
    pr = gm.params()
    want = {"loglik": outs[-1], "w": gm.w, "beta": pr["Bcoeff"], "tausq_inv": pr["tausq_inv"], "xb": pr["XB"]}
    gm.close()
    assert not np.array_equal(outs[-2], outs[-1])  # the last step is told apart from the one before it
    assert want["w"].shape == (625,) and np.any(want["w"] != 0) and not np.array_equal(want["w"], want["xb"])
    for k, v in want.items():
        assert np.array_equal(got[k], v), k


@pytest.mark.gpu
def test_product_arm_prints_one_json_line_with_the_contract_keys():
    """the CUDA arm on the smallest config (C1): ONE JSON line on stdout with every key the measurement contract names"""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "C1", "--steps", "20", "--warmup", "3"],
                       capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["metric"] == "mcmc_iterations_per_sec" and d["unit"] == "it/s" and d["n_gpus"] == 1 and d["steps"] == 20 and d["warmup"] == 3
    assert d["value"] > 0 and abs(d["ms_per_step"] * d["value"] - 1e3) < 1e-6 * 1e3 and d["higher_is_better"] is True
    assert d["scaling"] == "strong" and d["vs_baseline"] is None and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert set(d["config"]) == {"workload", "n", "q", "p", "blocks", "levels", "theta", "l2", "parallelism"} and d["config"]["workload"] == "C1"
    e = d["e2e"]
    assert e["value"] > 0 and e["unit"] == "it/s" and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] >= 8 * d["config"]["n"]
    assert d["gpu_launches"] > 20 * 20  # more than twenty kernels of this library per iteration
    rf = d["roofline"]
    assert rf["bound"] == "tensor" and rf["unit"] == "TFLOP/s" and rf["achieved"] > 0 and rf["peak"] > 0
    assert abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-12 and "traffic" in rf and 0 < rf["frac_executed"] <= rf["frac"]
    cb = d["cpu_baseline"]
    assert cb["value"] > 0 and cb["unit"] == "it/s" and cb["cores"] >= 1 and cb["kind"] == "port" and cb["sample"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert np.isfinite(d["parity_probe"]["loglik_w"])
