"""The reference arm of bench.py (`--impl reference`: the oracle port timed on the host cores) runs
without a GPU; its JSON line must carry the keys the measurement contract names. On the GPU,
`--dump-outputs` must write what the timed solve returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_reference(*extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1", *extra], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


@pytest.mark.parametrize("workload", ["c1", "c2", "sparse"])
def test_reference_arm_line(workload):
    # c2's own sample is n = m = 1000 (minutes of CPU work): the contract is checked on a smaller one
    d = run_reference("--workload", workload, *(["--cpu-size", "160"] if workload == "c2" else []))
    assert d["impl"] == "reference" and d["metric"] == "newton_step_ms" and d["unit"] == "ms"
    assert d["higher_is_better"] is False and d["n_gpus"] == 1 and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] == d["value"] and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    if workload in ("c1", "c2"):
        assert cb["blas3_gram"]["value"] > 0           # the BLAS-3 variant of the port beside the as-written one
    if workload == "c1":
        assert "extrapolat" not in cb["sample"]        # config 1 is measured at its own size
    if workload == "c2":
        # the work model is validated on a second sample size, and the bounded sample is declared
        assert cb["model_check"]["predicted_ms_per_step"] > 0 and cb["model_check"]["measured_ms_per_step"] > 0
        assert d["sample_steps"] == {"timed": 2, "warmup": 1} and "extrapolat" in d["config"]["measured_on"]


def test_other_ranks_of_the_reference_arm_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def run_b200(out_dir, *extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--no-cpu-baseline", "--dump-outputs", str(out_dir),
                          *extra], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


@pytest.mark.gpu
def test_dump_outputs_holds_the_result_of_the_timed_solve(tmp_path):
    import devlib
    import torch
    from harness import fill_workload
    args = ("--workload", "c1", "--steps", "2", "--warmup", "3", "--no-full-solve")
    d = run_b200(tmp_path / "a", *args)
    run_b200(tmp_path / "b", *args)
    names = ["iteration_log.npy", "y.npy"]
    assert sorted(os.listdir(tmp_path / "a")) == sorted(os.listdir(tmp_path / "b")) == names
    for name in names:                     # same arguments, same seeded inputs: the same bits
        a, b = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype == np.float64 and np.array_equal(a, b)
    y, log = np.load(tmp_path / "a" / "y.npy"), np.load(tmp_path / "a" / "iteration_log.npy")
    # warm-up + timed steps; the last row (columns by, cx) is the final iterate the line reports
    assert log.shape == (5, 8)
    assert log[-1, 4] == d["final"]["by"] and log[-1, 5] == d["final"]["cx"]
    # y is what the timed solve returns: the same 3 + 2 Newton steps on the same program, solved here (the warm-start
    # leg that follows in bench.py takes 2 more steps and returns another y)
    dev = devlib.product()
    P = dev.program()
    A, Cm, rb, rc = P.dense_lmi_storage(50, 100)
    bvec = fill_workload("random", 50, 100, rb, rc, A, Cm)
    torch.cuda.synchronize()
    del A, Cm
    _, y_here = P.maximize(bvec, dev.default_config(max_iterations=5, final_centering_steps=0, inv_sqrt_mu_max=1e12))
    assert y.shape == (100,) and np.abs(y - y_here).max() <= 1e-9 * np.abs(y_here).max()


@pytest.mark.gpu
def test_batched_workload_times_the_requested_lock_steps(tmp_path):
    import devlib
    from harness import Batch, add_cones, small_multicone_problem
    d = run_b200(tmp_path, "--workload", "c3", "--programs", "64", "--steps", "2", "--warmup", "3")
    assert d["steps"] == 2 and d["warmup"] == 3 and len(d["step_ms_per_step"]) == 2
    assert d["config"]["programs"] == 64 and d["solve_ms"] > 0
    y = np.load(tmp_path / "y.npy")
    # the timed solve is 3 warm-up + 2 timed lock steps of one solve: the same solve here returns the dumped y
    dev = devlib.product()
    programs, bs = [], []
    for p in range(64):
        cones, b = small_multicone_problem(1000 + p)
        P = dev.program()
        add_cones(P, cones)
        programs.append(P)
        bs.append(b)
    batch = Batch(dev, programs)
    _, y_here = batch.maximize(np.stack(bs), dev.default_config(max_iterations=5, final_centering_steps=0,
                                                                inv_sqrt_mu_max=1e12))
    assert len(batch.step_milliseconds()) == 5
    assert y.shape == (64, 40) and np.abs(y - y_here).max() <= 1e-9 * np.abs(y_here).max()
