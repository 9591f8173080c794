#!/usr/bin/env python
"""Benchmark of the conex-b200 Newton step (BASELINE.json metric: Newton-step ms and FP64 TFLOP/s
vs roofline).

  python bench.py --gpus N --steps K --warmup W          # B200 arm (one rank per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W  # CPU arm: the oracle port on the host cores

Default workload (config 2 of BASELINE.json, the one the metric is quoted on): MaxCut dual SDP on a
random graph, n = m = 2000, one dense PSD block driven through the dense-LMI path of the C ABI
(A_i = -e_i e_i^T stored as dense n x n matrices, 64 GB in HBM — far larger than the 126 MB L2, so
no L2 flush is needed between steps). A "step" is one full Newton step of CONEX_Maximize (assemble
H, factor, choose mu, solve, eigen-bound, geodesic update) at the running iterate; W + K steps run
inside one solve and every step is timed with CUDA events on the solver's stream. With N > 1 the same
step is sharded over the ranks (strong scaling). `--workload c5|c4|c1` selects the other single-block
configurations of BASELINE.json (large-m dense LMI, Lovasz theta, the small reference case).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# stdout carries exactly one JSON line: whatever NCCL logs (e.g. its version banner under
# NCCL_DEBUG=VERSION) goes to a file instead. Must be set before NCCL initialises.
os.environ.setdefault("NCCL_DEBUG_FILE", os.devnull)

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "newton_step_ms"
UNIT = "ms"


from conex_b200.workloads import device_view, fill_workload, lovasz_edges, structured_problem  # noqa: E402


def algorithmic_flops(n, m):
    """SURVEY.md §8(d): dense A_i, symmetry savings not credited."""
    k1 = 4.0 * m * n ** 3
    k2 = float(m) * (m + 1) * n ** 2
    k3 = m ** 3 / 3.0
    k78 = 12.7 * n ** 3
    return dict(k1=k1, k2=k2, k3=k3, k78=k78, tensor=k1 + k2 + k3 + k78)


WORKLOADS = {
    "c3": dict(kind="batched", n=20, m=40, programs=4096, cpu=dict(programs=128)),
    # structured path (SURVEY.md 8d caveat ii): the same operators given entry by entry through the
    # incremental API, assembled by gathers from W instead of matrix products
    "c2s": dict(kind="maxcut_entries", n=2000, m=2000, cpu=dict(n=400, m=400)),
    "c4s": dict(kind="lovasz_entries", n=500, m=10001, cpu=dict(n=100, m=401)),
    # chordal-sparse program (SURVEY.md 8 f4): 8 LMI cones (n = 60), each on 1500 private + 100 shared
    # variables through CONEX_AddSparseLMIConstraint -> block-arrow Schur complement of order 12100
    "sparse": dict(kind="arrow", n=60, m=12100, blocks=8, private=1500, shared=100,
                   cpu=dict(blocks=8, private=150, shared=10, n=20)),
    # cpu: the sample the --impl reference arm times (BASELINE.md 4: n = m = 1000); cpu_small: the 10-30 s sample of
    # the b200 arm's cpu_baseline leg; cpu_check: a second size that validates the per-phase work model
    "c2": dict(kind="maxcut", n=2000, m=2000, cpu=dict(n=1000, m=1000), cpu_small=dict(n=500, m=500),
               cpu_check=dict(n=400, m=400)),
    "c5": dict(kind="random", n=1000, m=20000, cpu=dict(n=120, m=600)),
    "c4": dict(kind="lovasz", n=500, m=10001, cpu=dict(n=100, m=401)),
    "c1": dict(kind="random", n=50, m=100, cpu=dict(n=50, m=100)),
}


def workload_shape(args):
    w = dict(WORKLOADS[args.workload])
    if args.n:
        w["n"] = args.n
        if w["kind"] in ("maxcut", "maxcut_entries"):
            w["m"] = args.n
    if args.m:
        w["m"] = args.m
    if args.programs and w["kind"] == "batched":
        w["programs"] = args.programs
    names = {"maxcut": "maxcut_sdp_n{n}_dense_lmi", "random": "dense_lmi_sdp_n{n}_m{m}",
             "lovasz": "lovasz_theta_n{n}_m{m}",
             "batched": "batched_small_sdp_{programs}x(3xpsd20+2xsoc10+lp40)_m40",
             "maxcut_entries": "maxcut_sdp_n{n}_entry_sparse", "lovasz_entries": "lovasz_theta_n{n}_m{m}_entry_sparse",
             "arrow": "block_arrow_{blocks}x(psd{n}_on_{private}_private+{shared}_shared_vars)_m{m}"}
    w["name"] = names[w["kind"]].format(**w)
    return w


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except ValueError:
                continue
            for name, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


def measure_fp64_peak():
    """cuBLAS DGEMM 8192^3 through torch, best of 5 — the FP64 roofline denominator.
    MEASURED_PEAKS.json carries only HBM and bf16 figures, so this one is measured live."""
    import torch
    n = 8192
    a = torch.randn((n, n), dtype=torch.float64, device="cuda")
    b = torch.randn((n, n), dtype=torch.float64, device="cuda")
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def _oracle_loader():
    """The CPU oracle (oracle/, test infrastructure) is loaded only by the cpu_baseline / --impl reference legs."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle_loader import oracle
    return oracle


def cpu_problem(kind, n, m):
    """(packed matrices (m x n^2, one column-major block per row), column-major C, b or None)."""
    from conex_b200.binding import fmat, pack_matrices
    from conex_b200.workloads import lovasz_theta_lmi, maxcut_lmi, random_dense_lmi
    if kind == "maxcut":
        if n <= 400:
            mats, Cm, b = maxcut_lmi(n, 2)
            return pack_matrices(mats), fmat(Cm), b
        # same instance family without the m dense numpy matrices (8 GB at n = 1000): packed buffer directly
        rng = np.random.Generator(np.random.PCG64(2))
        upper = np.triu(rng.random((n, n)) < 0.5, 1).astype(np.float64)
        adj = upper + upper.T
        A = np.zeros((n, n * n))
        A[np.arange(n), np.arange(n) * (n + 1)] = -1.0
        return A, fmat(-(np.diag(adj.sum(axis=1)) - adj) / 4.0), -np.ones(n)
    if kind == "lovasz":
        mats, Cm, b = lovasz_theta_lmi(n, m - 1, 4)
        return pack_matrices(mats), fmat(Cm), b
    mats, Cm = random_dense_lmi(n, m, 1)
    return pack_matrices(mats), fmat(Cm), None


def phase_model(n, m):
    """Work per phase used to extrapolate the CPU sample (SURVEY.md 8a): assembly 4mn^3 + m^2 n^2
    flop, factor m^3/3, each solve m^2, update/mu n^3-scale GEMMs + the mn^2 slack GEMV."""
    return dict(assemble=4.0 * m * n ** 3 + float(m) * m * n ** 2, factor=m ** 3 / 3.0, solve=float(m) * m,
                update=10.7 * n ** 3 + 2.0 * m * n ** 2, mu=4.0 * n ** 3 + 2.0 * m * n ** 2 + float(m) * m)


def cpu_sample(O, kind, ns, ms, total_steps, gram_variant):
    """One oracle solve of `total_steps` Newton steps on the (ns, ms) instance: per-step wall time and phases."""
    A, Cf, b = cpu_problem(kind, ns, ms)
    P = O.program()
    P.add_dense_lmi_packed(A, Cf, ns, ms)
    del A
    # 0: the Gram rows as conex computes them (m matrix-vector products, dense_lmi_constraint.cc:77-78);
    # 1: the same contraction as one BLAS-3 call — so that the GPU/CPU ratio is not inflated by the
    # reference's own BLAS-2 formulation (SURVEY.md 8d)
    O.lib.ORACLE_SetGramVariant(P.h, gram_variant)
    bb = P.feasible_objective() if b is None else b
    cfg = O.default_config(max_iterations=total_steps, final_centering_steps=0, inv_sqrt_mu_max=1e12)
    t0 = time.perf_counter()
    P.maximize(bb, cfg)
    wall = time.perf_counter() - t0
    its = max(P.status()["num_iterations"], 1)
    per = {k: v / its for k, v in P.phase_seconds().items()}
    return wall / its, its, per


def cpu_baseline(w, steps, warmup, threads=None, sample_key="cpu"):
    """Times the oracle port (reference algorithm as written, OpenBLAS underneath) on a reduced instance of the
    same workload and extrapolates each phase to the full shape with the work model above (the full operators,
    64-160 GB, do not fit the host; the as-written Gram alone would take many minutes per step). When the
    workload names a second sample size (`cpu_check`), the same model predicts the larger sample from the
    smaller one and the prediction is reported next to the measurement (`model_check`)."""
    oracle = _oracle_loader()
    O = oracle()
    cores = threads or os.cpu_count()
    O.lib.ORACLE_SetBlasThreads(cores)
    size = w.get(sample_key) or w["cpu"]
    ns, ms = size["n"], size["m"]
    total = warmup + steps
    full, small = phase_model(w["n"], w["m"]), phase_model(ns, ms)
    ratio = {k: full[k] / small[k] for k in full}
    same = (ns, ms) == (w["n"], w["m"])
    step3, its3, per3 = cpu_sample(O, w["kind"], ns, ms, total, 1)
    step0, its, per = cpu_sample(O, w["kind"], ns, ms, total, 0)
    full_s = sum(per[k] * ratio[k] for k in per)
    full3_s = sum(per3[k] * ratio[k] for k in per3)
    out = {
        "blas3_gram": {"value": (step3 if same else full3_s) * 1e3, "unit": UNIT, "sample_ms_per_step": step3 * 1e3,
                       "note": "same port with the Gram contraction as one BLAS-3 call instead of the reference's m "
                               "matrix-vector products"},
        "value": (step0 if same else full_s) * 1e3, "unit": UNIT, "cores": cores, "kind": "port",
        "sample": (f"oracle port (as-written Gram, OpenBLAS x{cores} threads) on {w['kind']} n={ns} m={ms}, "
                   f"{its} Newton steps, {step0 * 1e3:.1f} ms/step measured" +
                   ("" if same else "; value is the per-phase extrapolation to "
                    f"n={w['n']} m={w['m']} by the work model (" +
                    ", ".join(f"{k} x{ratio[k]:.0f}" for k in ratio) + ")")),
        "sample_ms_per_step": step0 * 1e3,
        "sample_phase_ms": {k: v * 1e3 for k, v in per.items()},
    }
    chk = w.get("cpu_check")
    if chk and (chk["n"], chk["m"]) != (ns, ms):
        # validate the model: predict THIS sample from a smaller one
        stepc, itsc, perc = cpu_sample(O, w["kind"], chk["n"], chk["m"], total, 0)
        tiny = phase_model(chk["n"], chk["m"])
        predicted = sum(perc[k] * small[k] / tiny[k] for k in perc)
        out["model_check"] = {
            "smaller_sample": f"n={chk['n']} m={chk['m']}: {stepc * 1e3:.1f} ms/step measured ({itsc} steps)",
            "predicted_ms_per_step": predicted * 1e3, "measured_ms_per_step": step0 * 1e3,
            "measured_over_predicted": step0 / predicted,
            "note": f"work model applied from n={chk['n']} to n={ns} (the same model carries n={ns} to n={w['n']}); a ratio "
                    "above 1 means the extrapolated value UNDERSTATES the CPU time (cache effects of the larger "
                    "operator), below 1 that it overstates it"}
    return out


# ---- BASELINE config 3: many small multi-cone programs, batched per GPU ----------------------------
def batched_flops_per_program_step(m=40, n=20, blocks=3):
    """Dense algorithmic flops of one Newton step of one program (SURVEY.md 8a): the PSD blocks
    dominate (4 m n^3 + m(m+1) n^2 each), + m^3/3 for the KKT Cholesky."""
    return blocks * (4.0 * m * n ** 3 + float(m) * (m + 1) * n ** 2) + m ** 3 / 3.0


def batched_bytes_per_program_step(m=40, n=20, blocks=3):
    """Algorithmic HBM bytes per program and step: three passes over the operator of the LMI blocks — the Schur system
    and the two slacks of a Newton step (SURVEY.md 8a). (The product reads less: the slack passes take the packed
    lower triangles, 2.5 instead of 3 x the operator; the scaled matrices never leave shared memory.)"""
    return blocks * (m + 1) * n * n * 8.0 * 3


def cpu_baseline_batched(w, count=None, workers=None):
    """The oracle port solving a bounded sample of the batch: every program is solved on its own, as the reference
    would, with one BLAS thread each (the matrices are 20 x 20) and `workers` host threads taking programs from the
    sample in parallel (default: every host core; the programs are independent, which is all the parallelism a CPU
    run of this workload has). Only the solves are timed."""
    from concurrent.futures import ThreadPoolExecutor
    from conex_b200.workloads import add_cones, small_multicone_problem
    oracle = _oracle_loader()
    O = oracle()
    O.lib.ORACLE_SetBlasThreads(1)
    workers = max(1, workers or (os.cpu_count() or 1))
    count = count or min(w["programs"], max(w["cpu"]["programs"], 256 * workers))   # ~20 core-seconds
    programs = []
    for p in range(count):
        cones, b = small_multicone_problem(1000 + p)
        P = O.program()
        add_cones(P, cones)
        programs.append((P, b))

    def solve(item):   # the library call releases the GIL
        item[0].maximize(item[1])
        return item[0].status()["num_iterations"]

    t0 = time.perf_counter()
    if workers == 1:
        steps = sum(solve(item) for item in programs)
    else:
        with ThreadPoolExecutor(max_workers=workers) as pool:
            steps = sum(pool.map(solve, programs))
    t_total = time.perf_counter() - t0
    per_program_step_ms = t_total / steps * 1e3    # wall time per program-step with all workers busy
    return {"value": per_program_step_ms * w["programs"], "unit": UNIT, "cores": workers, "kind": "port",
            "sample": f"oracle port solving {count} of the {w['programs']} programs, each on its own, {workers} at a "
                      f"time ({steps} Newton steps in {t_total:.2f} s of wall time = {per_program_step_ms:.3f} ms per "
                      f"program-step); value = that x {w['programs']} programs (one lock-step Newton step of the "
                      "whole batch)",
            "sample_solve_s": t_total, "sample_programs": count,
            "programs_per_s": count / t_total}


class Process:
    """One rank of the benchmark: device selection, torch.distributed (NCCL) for the plumbing, the product library
    and — on first use — its own NCCL communicator."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        import conex_b200.binding as devlib
        self.torch, self.dist, self.devlib = torch, dist, devlib
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.dev = devlib.product()
        self.L = self.dev.lib
        assert self.L.CONEXB200_DeviceAvailable() == 1, "no sm_100 device: conex-b200 has no CPU fallback"
        self._comm = False
        self.peak_tf = measure_fp64_peak()

    def communicator(self):
        if self.world > 1 and not self._comm:
            self.devlib.init_communicator(self.dev, self.rank, self.world)
            self._comm = True

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        if self.world == 1:
            return [float(v) for v in values]
        t = self.torch.tensor([float(v) for v in values], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.cpu().tolist()

    def sum_over_ranks(self, values):
        if self.world == 1:
            return [float(v) for v in values]
        t = self.torch.tensor([float(v) for v in values], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return t.cpu().tolist()

    def release(self):
        import gc
        gc.collect()
        self.torch.cuda.empty_cache()

    def close(self):
        if self._comm:
            self.L.CONEXB200_CommDestroy()
        if self.world > 1:
            self.dist.destroy_process_group()


def measure_h2d_rate(torch, nbytes=1 << 30):
    """Pinned host -> device copy rate (GB/s), for the one-time cost of CONEX_AddDenseLMIConstraint with HOST matrices."""
    try:
        h = torch.empty(nbytes // 8, dtype=torch.float64).pin_memory()
        d = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
        d.copy_(h, non_blocking=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        d.copy_(h, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        rate = nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9
        del h, d
        torch.cuda.empty_cache()
        return rate
    except Exception:
        return None


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(directory, arrays):
    """--dump-outputs: each array as DIR/<name>.npy in float64, so that two builds run with the same arguments (and
    therefore the same seeded inputs) can be compared output for output. An array larger than its share of the 64 MB
    budget is replaced by a fixed, seeded sample of its rows."""
    os.makedirs(directory, exist_ok=True)
    share = DUMP_BUDGET_BYTES // max(len(arrays), 1)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if a.nbytes > share:
            rows = max(1, share // (a.nbytes // a.shape[0]))
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], rows, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


def log_array(log):
    """Program.iteration_log() as an (iterations x 8) array, columns in the order of its keys."""
    return np.array([list(row.values()) for row in log])


def hbm_peak():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6534.8, "B200_PROFILING.md fallback 6534.8 GB/s"


def batched_bench(proc, args, w, steps, warmup, cpu_leg, outputs=None):
    """BASELINE config 3 on this process' share of the programs; returns the JSON dict on rank 0, None elsewhere.
    `outputs` (a dict) receives y of the timed solve, all programs."""
    from conex_b200.binding import Batch
    from conex_b200.workloads import add_cones, small_multicone_problem
    torch, dev, L, world, rank = proc.torch, proc.dev, proc.L, proc.world, proc.rank
    total_programs = w["programs"]
    lo = total_programs * rank // world
    hi = total_programs * (rank + 1) // world
    t_setup = time.perf_counter()
    programs, bs = [], []
    for p in range(lo, hi):
        cones, b = small_multicone_problem(1000 + p)
        P = dev.program()
        add_cones(P, cones)
        programs.append(P)
        bs.append(b)
    batch = Batch(dev, programs)
    b = np.stack(bs)
    del programs
    setup_s = time.perf_counter() - t_setup

    # W warm-up + K timed lock steps in one solve, as the dense path times its Newton steps; without final centering
    # every program takes a full Newton step in each of them
    total = warmup + steps
    cfg = dev.default_config(max_iterations=total, final_centering_steps=0, inv_sqrt_mu_max=1e12)
    proc.barrier()
    sampler = ClockSampler(proc.local_rank)
    sampler.start()
    launches0 = L.CONEXB200_LaunchCount()
    _, y = batch.maximize(b, cfg)
    torch.cuda.synchronize()
    launches = L.CONEXB200_LaunchCount() - launches0
    clocks = sampler.stop()
    step_ms = batch.step_milliseconds()
    assert len(step_ms) == total, f"expected {total} lock steps, ran {len(step_ms)}"
    timed = step_ms[warmup:]
    its = batch.results()[0]
    if outputs is not None:
        if world > 1:
            parts = [None] * world
            proc.dist.all_gather_object(parts, y)
            y = np.concatenate(parts)
        outputs["y"] = y

    # whole-solve throughput: a cold-start solve with the DEFAULT configuration, run to termination
    proc.barrier()
    t0 = time.perf_counter()
    solved, _ = batch.maximize(b, dev.default_config())
    torch.cuda.synchronize()
    e2e_wall = time.perf_counter() - t0
    solve_steps = len(batch.step_milliseconds())
    dev_ms = batch.milliseconds()
    timed_ms = float(timed.sum())
    dev_ms, e2e_ms, timed_ms = proc.max_over_ranks([dev_ms, e2e_wall * 1e3, timed_ms])
    program_steps, nsolved, nprog = proc.sum_over_ranks([float(np.clip(its - warmup, 0, steps).sum()),
                                                         float(solved.sum()), float(hi - lo)])
    nsolved, nprog = int(nsolved), int(nprog)
    del batch
    proc.release()
    if rank != 0:
        return None
    mean_step_ms = timed_ms / steps
    flops = batched_flops_per_program_step() * program_steps
    bytes_ = batched_bytes_per_program_step() * program_steps
    peak, peak_src = hbm_peak()
    line = {
        "metric": METRIC, "value": mean_step_ms, "unit": UNIT, "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": mean_step_ms, "higher_is_better": False, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": w["name"], "programs": nprog, "m": 40,
                   "path": "CONEXB200_BatchMaximize: all programs advance one Newton step per launch set",
                   "l2": "cone data 1.6 GB per step vs 126 MB L2: no flush",
                   "multi_gpu": (f"programs partitioned over {world} ranks, no collective" if world > 1 else "n/a"),
                   "step": "one lock-step Newton step of the whole batch (mean over the K timed steps that follow W "
                           "warm-up steps of one solve without final centering)"},
        "step_ms_per_step": [round(float(v), 4) for v in timed],
        "solve_ms": dev_ms, "solve_lock_steps": solve_steps, "programs_per_s": nprog / (dev_ms * 1e-3),
        "programs_solved": nsolved, "program_steps": program_steps,
        "step_tflops_fp64": flops / (timed_ms * 1e-3) / 1e12,
        "roofline": {"bound": "hbm", "kernel": "whole lock step of the batch: PsdSchurMma2Kernel (DMMA, 66 % pipe-active under "
                                               "ncu, profiles/r02_m_c3_schur_ncu_full.txt) + the eigen-bound / step kernels",
                     "achieved": bytes_ / (timed_ms * 1e-3) / 1e9, "peak": peak * world, "unit": "GB/s",
                     "frac": bytes_ / (timed_ms * 1e-3) / 1e9 / (peak * world), "peak_source": peak_src,
                     "note": "time of the timed lock steps, all kernels; the same work is 2 flop/byte-balanced: "
                             f"{flops / (timed_ms * 1e-3) / 1e12:.2f} TFLOP/s FP64 vs {proc.peak_tf:.1f} TFLOP/s cuBLAS DGEMM",
                     "traffic": None},
        "e2e": {"value": e2e_ms / max(solve_steps, 1), "unit": UNIT, "solve_ms": e2e_ms,
                "h2d_bytes_per_step": 8.0 * 40 * nprog / max(solve_steps, 1) + 8.0 * 6 * nprog,
                "d2h_bytes_per_step": 8.0 * 40 * nprog / max(solve_steps, 1) + 8.0 * (2 * 6 * 4 + 6) * nprog,
                "note": "default-configuration CONEXB200_BatchMaximize from host b to host y (wall clock / lock steps)"},
        "gpu_launches": int(launches), "clocks": clocks, "setup_s": setup_s,
    }
    if cpu_leg:
        line["cpu_baseline"] = cpu_baseline_batched(w)
    return line


def run_b200_batched(args):
    proc = Process()
    if args.small_psd_mma >= 0:
        proc.L.cxb_set_small_psd_mma(args.small_psd_mma)
    if args.small_team_mode >= 0:
        proc.L.cxb_set_small_team_mode(args.small_team_mode)
    if args.small_cone_threads > 0:
        proc.L.cxb_set_small_cone_threads(args.small_cone_threads)
    if args.small_fused_launches >= 0:
        proc.L.cxb_set_small_fused_launches(args.small_fused_launches)
    outputs = {} if args.dump_outputs else None
    line = batched_bench(proc, args, workload_shape(args), args.steps, args.warmup, cpu_leg=not args.no_cpu_baseline,
                         outputs=outputs)
    if line is not None:
        print(json.dumps(line))
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
    proc.close()


# ---- structured path: entry-sparse operators through the incremental API ---------------------------
def structured_flops(n, m):
    """Own algorithmic count of the structured step: K3 + two W.S GEMMs + W C W (4 n^3) + K8."""
    return m ** 3 / 3.0 + 4.0 * n ** 3 + 4.0 * n ** 3 + 8.7 * n ** 3


def run_b200_structured(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import conex_b200.binding as devlib
    dev = devlib.product()
    L = dev.lib
    assert L.CONEXB200_DeviceAvailable() == 1, "no sm_100 device: conex-b200 has no CPU fallback"
    w = workload_shape(args)
    n, m = w["n"], w["m"]
    peak_tf = measure_fp64_peak()
    t_setup = time.perf_counter()
    entries, Cm, b = structured_problem(w)
    if world > 1:
        devlib.init_communicator(dev, rank, world)
    configure_cholesky(L, args)
    P = dev.program(m)
    if world > 1:
        # every rank builds the same program and solves in lock step: the entry-sparse assembly and
        # the n-sized phases are replicated, the Cholesky of the m x m Schur complement is distributed
        L.CONEXB200_SetCollective(P.h, 1)
    cid = C.c_int(-1)
    assert L.CONEX_NewLinearMatrixInequality(P.h, n, 1, C.byref(cid)) == 0
    for (v, r, c, val) in entries:
        assert L.CONEX_UpdateLinearOperator(P.h, cid.value, float(val), v, r, c, 0) == 0
    rr, cc = np.nonzero(np.tril(Cm))
    for r, c in zip(rr.tolist(), cc.tolist()):
        L.CONEX_UpdateAffineTerm(P.h, cid.value, float(Cm[r, c]), r, c, 0)
    P.cone_shapes.append((n, n))
    setup_s = time.perf_counter() - t_setup
    total = args.warmup + args.steps
    cfg = dev.default_config(max_iterations=total, final_centering_steps=0, inv_sqrt_mu_max=1e12)
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = L.CONEXB200_LaunchCount()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    solved, y = P.maximize(b, cfg)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    launches = L.CONEXB200_LaunchCount() - launches0
    outputs = {"y": y, "iteration_log": log_array(P.iteration_log())} if args.dump_outputs else None
    assert L.CONEXB200_ConstraintIsEntrySparse(P.h, cid.value) == 1
    its = P.status()["num_iterations"]
    ms = np.zeros(1)
    step_ms, phases = [], []
    for i in range(its):
        L.CONEXB200_GetIterationMilliseconds(P.h, i, ms.ctypes.data_as(C.POINTER(C.c_double)))
        step_ms.append(float(ms[0]))
        ph = np.zeros(5)
        L.CONEXB200_GetIterationPhaseMilliseconds(P.h, i, ph.ctypes.data_as(C.POINTER(C.c_double)))
        phases.append(ph)
    timed = np.array(step_ms[args.warmup:])
    ph_timed = np.array(phases[args.warmup:]).mean(axis=0)
    # e2e: a complete solve with the default configuration, host b -> host y
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    solved2, y2 = P.maximize(b, dev.default_config())
    torch.cuda.synchronize()
    solve_wall = time.perf_counter() - t0
    solve_its = P.status()["num_iterations"]
    log = P.iteration_log()
    clocks = sampler.stop()
    value = float(timed.mean())
    if world > 1:
        t = torch.tensor([value, solve_wall] + ph_timed.tolist(), dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        value, solve_wall = float(t[0]), float(t[1])
        ph_timed = t[2:].cpu().numpy()
        L.CONEXB200_CommDestroy()
        dist.destroy_process_group()
        if rank != 0:
            return
    fl = structured_flops(n, m)
    upd = float(ph_timed[4])
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": value, "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": w["name"], "n": n, "m": m, "cholesky": cholesky_note(args, world, m),
                   "path": "incremental LMI (CONEX_NewLinearMatrixInequality + CONEX_UpdateLinearOperator), entry-sparse "
                           f"operator ({len(entries)} stored entries instead of {8e-9 * m * n * n:.1f} GB of dense matrices)",
                   "l2": "working set W, WS, H (tens of MB) is L2-resident by nature of the path; steps are not separated "
                         "by a flush",
                   "multi_gpu": (f"collective program on {world} ranks: Cholesky of the {m} x {m} Schur complement in 1-D "
                                 "block-cyclic block columns with NCCL panel broadcasts; assembly, solves, eigen-bounds and "
                                 "the geodesic update replicated") if world > 1 else "n/a"},
        "phase_ms": dict(zip(["assemble", "factor", "mu", "solve", "update"], ph_timed.tolist())),
        "step_tflops_fp64": fl / (value * 1e-3) / 1e12,
        "roofline": {"bound": "tensor", "kernel": "update phase: W.S GEMM, Taylor exponential GEMM chain, W <- E W (K7 + K8)",
                     "achieved": (2.0 + 8.0 + 2.0) * n ** 3 / (upd * 1e-3) / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": (2.0 + 8.0 + 2.0) * n ** 3 / (upd * 1e-3) / 1e12 / peak_tf,
                     "peak_source": "cuBLAS DGEMM 8192^3 measured live in this run",
                     "note": "own algorithmic count of the structured step (never the dense flops): the update phase "
                             "executes 6 n x n x n GEMMs; the phase is launch/latency-bound at this size (Lanczos)",
                     "traffic": None},
        "e2e": {"value": solve_wall * 1e3 / max(solve_its, 1), "unit": UNIT, "solve_ms": solve_wall * 1e3,
                "solve_iterations": solve_its, "solved": int(solved2),
                "h2d_bytes_per_step": 8.0 * m / max(solve_its, 1), "d2h_bytes_per_step": 8.0 * m / max(solve_its, 1) + 8.0 * (n + 12) * 2,
                "note": "complete CONEX_Maximize solve (default configuration) from host b to host y, wall clock / iterations"},
        "gpu_launches": int(launches), "clocks": clocks, "setup_s": setup_s, "first_solve_wall_s": wall,
        "final": {"by": log[-1]["by"], "cx": log[-1]["cx"], "mu": log[-1]["mu"]},
    }
    print(json.dumps(line))
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)


def arrow_flops(blocks, private, shared, n):
    """Own algorithmic count of one Newton step of the block-arrow program: per cone the dense-LMI
    assembly on its mc = private + shared variables, the multifrontal factorisation (leaf fronts
    s = private, p = shared; root s = private + shared) and the n-sized phases."""
    mc = private + shared
    asm = blocks * (4.0 * mc * n ** 3 + float(mc) * (mc + 1) * n ** 2)
    leaf = private ** 3 / 3.0 + float(private) ** 2 * shared + float(private) * shared ** 2
    fac = (blocks - 1) * leaf + mc ** 3 / 3.0
    return dict(assemble=asm, factor=fac, rest=blocks * 12.7 * n ** 3)


def run_b200_sparse(args):
    """Chordal-sparse program through CONEX_AddSparseLMIConstraint / CONEX_Maximize: the device picks the
    multifrontal KKT solver; the dense solver (one supernode of order m) is timed beside it."""
    import torch
    import conex_b200.binding as devlib
    from conex_b200.workloads import block_arrow_program
    dev = devlib.product()
    L = dev.lib
    assert L.CONEXB200_DeviceAvailable() == 1, "no sm_100 device: conex-b200 has no CPU fallback"
    assert int(os.environ.get("WORLD_SIZE", "1")) == 1, "the multifrontal solver is single-GPU (replicas only)"
    L.CONEXB200_SetKKTSolverKind.argtypes = [C.c_void_p, C.c_int]
    L.CONEXB200_SetKKTSolverKind.restype = None
    w = workload_shape(args)
    blocks, private, shared, n = w["blocks"], w["private"], w["shared"], w["n"]
    peak_tf = measure_fp64_peak()
    t_setup = time.perf_counter()
    m, cones = block_arrow_program(blocks, private, shared, n, seed=11)
    setup_s = time.perf_counter() - t_setup
    total = args.warmup + args.steps
    out = {}
    sampler = ClockSampler(0)
    sampler.start()
    for kind, name in ((1, "dense"), (0, "auto")):
        P = dev.program(m)
        L.CONEXB200_SetKKTSolverKind(P.h, kind)
        for mats, Cm, variables in cones:
            P.add_dense_lmi(mats, Cm, variables)
        b = P.feasible_objective()
        cfg = dev.default_config(max_iterations=total, final_centering_steps=0, inv_sqrt_mu_max=1e12)
        launches0 = L.CONEXB200_LaunchCount()
        _, y = P.maximize(b, cfg)
        torch.cuda.synchronize()
        launches = L.CONEXB200_LaunchCount() - launches0
        if name == "auto" and args.dump_outputs:
            outputs = {"y": y, "iteration_log": log_array(P.iteration_log())}
        its = P.status()["num_iterations"]
        assert its == total, f"expected {total} Newton steps, ran {its}"
        ms = np.zeros(1)
        step_ms, phases = [], []
        for i in range(its):
            L.CONEXB200_GetIterationMilliseconds(P.h, i, ms.ctypes.data_as(C.POINTER(C.c_double)))
            step_ms.append(float(ms[0]))
            ph = np.zeros(5)
            L.CONEXB200_GetIterationPhaseMilliseconds(P.h, i, ph.ctypes.data_as(C.POINTER(C.c_double)))
            phases.append(ph)
        # e2e: a complete solve with the default configuration, host b -> host y
        t0 = time.perf_counter()
        solved, y = P.maximize(b, dev.default_config())
        torch.cuda.synchronize()
        solve_wall = time.perf_counter() - t0
        out[name] = dict(step=float(np.mean(step_ms[args.warmup:])), phases=np.array(phases[args.warmup:]).mean(axis=0),
                         supernodes=L.CONEXB200_GetNumberOfSupernodes(P.h), solved=int(solved),
                         solve_ms=solve_wall * 1e3, solve_its=P.status()["num_iterations"], launches=int(launches),
                         by=P.iteration_log()[-1]["by"])
    clocks = sampler.stop()
    a, d = out["auto"], out["dense"]
    fl = arrow_flops(blocks, private, shared, n)
    fac_ms = float(a["phases"][1])
    line = {
        "metric": METRIC, "value": a["step"], "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": a["step"], "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": w["name"], "n": n, "m": m,
                   "path": f"{blocks} dense LMI cones on variable subsets (CONEX_AddSparseLMIConstraint); KKT solver chosen by "
                           f"the library: {a['supernodes']} supernodes (multifrontal)" if a["supernodes"] > 1 else "dense",
                   "l2": "operators 8 x 46 MB + fronts 150 MB vs 126 MB L2: no flush", "multi_gpu": "n/a"},
        "phase_ms": dict(zip(["assemble", "factor", "mu", "solve", "update"], [float(v) for v in a["phases"]])),
        "dense_kkt_solver": {"newton_step_ms": d["step"], "supernodes": d["supernodes"],
                             "phase_ms": dict(zip(["assemble", "factor", "mu", "solve", "update"], [float(v) for v in d["phases"]])),
                             "final_by": d["by"]},
        "roofline": {"bound": "tensor", "kernel": "multifrontal factorisation (PotrfDiagBlockedKernel / TrsmPanelKernel / DgemmKernel per front)",
                     "achieved": fl["factor"] / (fac_ms * 1e-3) / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": fl["factor"] / (fac_ms * 1e-3) / 1e12 / peak_tf,
                     "peak_source": "cuBLAS DGEMM 8192^3 measured live in this run",
                     "algorithmic_flops_per_step": fl["factor"],
                     "note": "own algorithmic count (sum over fronts of s^3/3 + s^2 p + s p^2); fronts of order 1500-1600 are "
                             "panel-latency-bound, the gain over the dense solver is the 50x smaller flop count",
                     "traffic": None},
        "e2e": {"value": a["solve_ms"] / max(a["solve_its"], 1), "unit": UNIT, "solve_ms": a["solve_ms"],
                "solve_iterations": a["solve_its"], "solved": a["solved"],
                "h2d_bytes_per_step": 8.0 * m / max(a["solve_its"], 1),
                "d2h_bytes_per_step": 8.0 * m / max(a["solve_its"], 1) + blocks * 8.0 * (n + 12) * 2,
                "note": "complete CONEX_Maximize solve (default configuration) from host b to host y, wall clock / iterations"},
        "gpu_launches": a["launches"], "clocks": clocks, "setup_s": setup_s,
        "final": {"by": a["by"]},
    }
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_sparse(w)
    print(json.dumps(line))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)


def cpu_baseline_sparse(w):
    """The oracle port (dense KKT matrix, like its stand-in for kkt_solver.cc) on a reduced block-arrow
    program; reported per step as measured — no extrapolation (the reference's own solver is
    supernodal, so a dense extrapolation to order 12100 would overstate its cost)."""
    oracle = _oracle_loader()
    from conex_b200.workloads import block_arrow_program
    O = oracle()
    cores = os.cpu_count()
    O.lib.ORACLE_SetBlasThreads(cores)
    c = w["cpu"]
    m, cones = block_arrow_program(c["blocks"], c["private"], c["shared"], c["n"], seed=11)
    P = O.program(m)
    for mats, Cm, variables in cones:
        P.add_dense_lmi(mats, Cm, variables)
    b = P.feasible_objective()
    t0 = time.perf_counter()
    P.maximize(b, O.default_config())
    wall = time.perf_counter() - t0
    its = max(P.status()["num_iterations"], 1)
    return {"value": wall / its * 1e3, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"oracle port on a reduced block-arrow program ({c['blocks']} cones of order {c['n']} on {c['private']} "
                      f"private + {c['shared']} shared variables, KKT order {m}), {its} Newton steps, measured per step, "
                      "not extrapolated"}


def configure_cholesky(L, args):
    """--replicated-cholesky: factor on every rank (the A/B arm of the multi-GPU Cholesky);
    --cholesky-block: block-column width of the distributed factorisation."""
    if args.replicated_cholesky:
        L.CONEXB200_SetDistributedCholesky(2 ** 30, 0)
    elif args.cholesky_block:
        L.CONEXB200_SetDistributedCholesky(-1, args.cholesky_block)


def cholesky_note(args, world, order):
    if world == 1:
        return "single GPU"
    if args.replicated_cholesky or order < 4096:
        return "replicated on every rank"
    return f"distributed: 1-D block-cyclic block columns of {args.cholesky_block or 512}, NCCL panel broadcasts"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = workload_shape(args)
    if w["kind"] in ("maxcut_entries", "lovasz_entries"):
        w = dict(w, kind=w["kind"].split("_")[0])
    if w["kind"] == "arrow":
        cb = cpu_baseline_sparse(w)
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT,
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": cb["value"], "higher_is_better": False, "scaling": "strong",
                          "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                          "config": {"workload": w["name"], "measured_on": "reduced program, see cpu_baseline.sample"},
                          "cpu_baseline": cb,
                          "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                                  "d2h_bytes_per_step": 0}}))
        return
    if w["kind"] == "batched":
        cb = cpu_baseline_batched(w)
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT,
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": cb["value"], "higher_is_better": False, "scaling": "strong",
                          "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                          "config": {"workload": w["name"], "programs": w["programs"]}, "cpu_baseline": cb,
                          "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                                  "d2h_bytes_per_step": 0}}))
        return
    if args.cpu_size:
        w["cpu"] = dict(n=args.cpu_size, m=args.cpu_size)
        w["cpu_check"] = dict(n=max(args.cpu_size // 2, 8), m=max(args.cpu_size // 2, 8))
    # a step of the CPU sample takes 20-40 s at n = m = 1000: the run is bounded to 1 warm-up + 2 timed steps whatever
    # K and W ask for (the line still carries the requested K / W, `sample_steps` what was run)
    k_cpu, w_cpu = min(args.steps, 2), min(args.warmup, 1)
    cb = cpu_baseline(w, k_cpu, w_cpu)
    same = (w["cpu"]["n"], w["cpu"]["m"]) == (w["n"], w["m"])
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "sample_steps": {"timed": k_cpu, "warmup": w_cpu},
        "ms_per_step": cb["value"],
        "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": w["name"], "n": w["n"], "m": w["m"],
                   "measured_on": ("the full shape" if same else
                                   f"n={w['cpu']['n']} m={w['cpu']['m']} sample of the same workload (the full operator, "
                                   f"{8e-9 * w['m'] * w['n'] ** 2:.0f} GB, and its as-written Gram do not fit a host run of minutes); "
                                   "value = per-phase extrapolation by the work model, validated on a second size in "
                                   "cpu_baseline.model_check")},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# DRAM traffic (dram__bytes_read.sum + dram__bytes_write.sum) of the DgemmKernel launches of ONE assembly phase of
# the C2 Newton step, per assembly form, from `ncu --set full` captures (per launch x launches per phase);
# None until a capture of that form exists.
ASSEMBLY_TRAFFIC_C2 = {
    1: dict(bytes=61 * (2.381e9 + 1.998e9) + 1.3545e12, source="profiles/r01_d_c2_dgemm_ncu_full.txt (classic form: 61 panels x "
            "(K1a 2.38 GB + K1b 2.00 GB) + K2 1354.5 GB of tile re-reads at 36 % L2 hit)"),
    3: dict(bytes=60 * (1.348e9 + 1.027e9 + 0.648e9 + 0.547e9) + (0.861e9 + 0.644e9 + 0.419e9 + 0.340e9) + 400.12e9,
            source="profiles/r02_e_c2_symmetric_assembly_ncu_full.txt (symmetric form: 60 panels of 33 matrices x (K1a A_i L 2.38 GB "
                   "+ K1b L^T T with packed store 1.20 GB) + one of 21 + K2 packed Gram 400 GB read at 58 % L2 hit for 35 GB of "
                   "operand; all three kernels run at 91-92 % DMMA-pipe active, i.e. tensor-bound; algorithmic minimum 64 GB of A "
                   "read + 35 GB of packed matrices written and read once)"),
}
FORM_NAMES = {0: "undecided", 1: "classic (W A_i W kept)", 2: "row panels (classic, streamed)", 3: "symmetric (packed L^T A_i L)",
              4: "entry-sparse gathers"}


def executed_assembly_flops(form, n, m):
    """What the assembly kernels of each form execute (not the dense algorithmic count): symmetric form — A_i L with
    the zeros of L skipped (n^3), lower tiles of L^T (A_i L) (n^3 / 3), Gram over the packed length Kp ~ 0.54 n^2 on the
    lower triangle of the (m + 2)-row operand; classic — A_i W (2 n^3), lower half of W (A_i W) mirrored (n^3), Gram
    m (m + 1) n^2."""
    if form == 3:
        t = (n + 63) // 64
        kp = t * (t + 1) // 2 * 4096
        return (4.0 / 3.0) * (m + 1) * n ** 3 + float(kp) * (m + 2) * (m + 3)
    return 3.0 * (m + 1) * n ** 3 + float(m) * (m + 1) * n ** 2


def dense_bench(proc, args, w, steps, warmup, full_solve, cpu_leg, outputs=None):
    """One dense-LMI workload (c1 / c2 / c4 / c5) on all ranks; returns the JSON dict on rank 0, None elsewhere.
    `outputs` (a dict) receives y and the iteration log of the timed solve."""
    torch, dist, dev, L, world, rank = proc.torch, proc.dist, proc.dev, proc.L, proc.world, proc.rank
    n, m = w["n"], w["m"]
    fl = algorithmic_flops(n, m)

    # ---- build the program with device-resident data (N > 1: this rank's shard of the rows) ----
    t_setup = time.perf_counter()
    proc.communicator()
    configure_cholesky(L, args)
    P = dev.program()
    if args.assembly_mode:
        L.CONEXB200_SetAssemblyMode(P.h, args.assembly_mode)
    if args.no_peer_memory:
        L.CONEXB200_SetPeerMemoryExchange(P.h, 0)
    try:
        A, Cm, rb, rc = P.dense_lmi_storage(n, m, world, rank)
    except AssertionError as e:
        return {"error": f"{w['name']}: {e}"} if rank == 0 else None
    b_local = fill_workload(w["kind"], n, m, rb, rc, A, Cm)
    torch.cuda.synchronize()
    del A, Cm
    torch.cuda.empty_cache()
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, b_local)
        b = np.concatenate(parts)
    else:
        b = b_local
    setup_s = time.perf_counter() - t_setup

    total = warmup + steps
    cfg = dev.default_config(max_iterations=total, final_centering_steps=0, inv_sqrt_mu_max=1e12)
    proc.barrier()
    sampler = ClockSampler(proc.local_rank)
    sampler.start()
    t0 = time.perf_counter()
    solved, y = P.maximize(b, cfg)
    torch.cuda.synchronize()
    wall_cold = time.perf_counter() - t0
    its = P.status()["num_iterations"]
    assert its == total, f"expected {total} Newton steps, ran {its}"
    ms = np.zeros(1)
    step_ms, phases = [], []
    for i in range(its):
        L.CONEXB200_GetIterationMilliseconds(P.h, i, ms.ctypes.data_as(C.POINTER(C.c_double)))
        step_ms.append(float(ms[0]))
        ph = np.zeros(5)
        L.CONEXB200_GetIterationPhaseMilliseconds(P.h, i, ph.ctypes.data_as(C.POINTER(C.c_double)))
        phases.append(ph)
    timed = np.array(step_ms[warmup:])
    ph_timed = np.array(phases[warmup:]).mean(axis=0)
    log = P.iteration_log()
    if outputs is not None:
        outputs["y"] = y
        outputs["iteration_log"] = log_array(log)
    form = L.CONEXB200_GetAssemblyForm(P.h, 0)
    shard = np.zeros(4)
    has_shard = L.CONEXB200_GetShardPhaseMilliseconds(P.h, 0, shard.ctypes.data_as(C.POINTER(C.c_double))) == 1

    # ---- e2e: exactly K more Newton steps through the C ABI with host buffers (warm start) ----
    cfg_e2e = dev.default_config(max_iterations=steps, final_centering_steps=0,
                                 inv_sqrt_mu_max=1e12, initialization_mode=1)
    launches0 = L.CONEXB200_LaunchCount()
    proc.barrier()
    t0 = time.perf_counter()
    P.maximize(b, cfg_e2e)
    torch.cuda.synchronize()
    e2e_wall = time.perf_counter() - t0
    launches = L.CONEXB200_LaunchCount() - launches0
    e2e_its = max(P.status()["num_iterations"], 1)
    e2e_step_ms = []
    for i in range(e2e_its):
        L.CONEXB200_GetIterationMilliseconds(P.h, i, ms.ctypes.data_as(C.POINTER(C.c_double)))
        e2e_step_ms.append(round(float(ms[0]), 3))
    clocks = sampler.stop()

    # ---- IPM solve time: a cold-start solve with the DEFAULT configuration, run to termination ----
    solve = None
    if full_solve:
        proc.barrier()
        t0 = time.perf_counter()
        s_full, y_full = P.maximize(b, dev.default_config())
        torch.cuda.synchronize()
        solve_wall = time.perf_counter() - t0
        flog = P.iteration_log()
        solve_its = P.status()["num_iterations"]
        dev_total = 0.0
        for i in range(solve_its):
            L.CONEXB200_GetIterationMilliseconds(P.h, i, ms.ctypes.data_as(C.POINTER(C.c_double)))
            dev_total += float(ms[0])
        solve_wall_max, dev_total = proc.max_over_ranks([solve_wall, dev_total])
        solve = {"solve_ms": solve_wall_max * 1e3, "solve_device_ms": dev_total, "solve_iterations": solve_its,
                 "solved": int(s_full), "by": flog[-1]["by"], "cx": flog[-1]["cx"], "mu": flog[-1]["mu"],
                 "note": "CONEX_Maximize, default CONEX_SolverConfiguration, cold start, host b -> host y (wall clock, "
                         "max over ranks)"}

    value = float(timed.mean())
    e2e_ms = e2e_wall * 1e3 / e2e_its
    red = proc.max_over_ranks([value, e2e_ms] + ph_timed.tolist() + shard.tolist())
    value, e2e_ms, ph_timed, shard = red[0], red[1], np.array(red[2:7]), red[7:]
    del P
    proc.release()
    if rank != 0:
        return None

    asm_ms = float(ph_timed[0])
    dense_flops = fl["k1"] + fl["k2"]
    exec_flops = executed_assembly_flops(form, n, m)
    achieved = exec_flops / (asm_ms * 1e-3) / 1e12
    peak = proc.peak_tf * world
    traffic = ASSEMBLY_TRAFFIC_C2.get(form) if (w["kind"], n, m, world) == ("maxcut", 2000, 2000, 1) else None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": value, "higher_is_better": False, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": w["name"], "n": n, "m": m,
                   "path": f"dense-LMI path of the C ABI (dense A_i, {8e-9 * m * n * n:.1f} GB resident)",
                   "assembly_form": FORM_NAMES.get(form, str(form)),
                   "l2": f"inputs ({8e-9 * m * n * n:.1f} GB) vs 126 MB L2: " +
                         ("no flush needed" if 8.0 * m * n * n > 4 * 126e6 else "L2-resident workload"),
                   "multi_gpu": (f"one Newton step sharded over {world} ranks: constraint matrices and the rows "
                                 "of H partitioned 1-D (K1/K2/K6 sharded, peers' scaled matrices pulled from "
                                 "peer memory over NVLink" + (" [A/B: ncclSend/ncclRecv]" if args.no_peer_memory else "") +
                                 ", H by all-reduce); Cholesky " + cholesky_note(args, world, m) +
                                 "; solve/eigen-bound/geodesic update replicated") if world > 1 else "n/a"},
        "newton_steps_per_s": 1e3 / value,
        "step_tflops_fp64": fl["tensor"] / (value * 1e-3) / 1e12,
        "phase_ms": dict(zip(["assemble", "factor", "mu", "solve", "update"], ph_timed.tolist())),
        "phase_ms_per_step": [[round(float(v), 3) for v in ph] for ph in phases[warmup:]],
        "roofline": {
            "bound": "tensor", "kernel": "DgemmKernel (K1 scaling GEMMs + K2 Gram, Schur assembly phase)",
            "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "peak_source": "cuBLAS DGEMM 8192^3 measured live in this run, times n_gpus (MEASURED_PEAKS.json has no FP64 "
                           "figure; nominal B200 FP64 tensor = 37 TFLOP/s)",
            "flops_counted": "EXECUTED flops of the assembly form in use (executed_flops_per_step) over the CUDA-event time "
                             "of the assembly phase — a hardware fraction",
            "executed_flops_per_step": exec_flops,
            "algorithmic_flops_per_step": dense_flops,
            "algorithmic_speedup": dense_flops / exec_flops,
            "achieved_on_algorithmic_flops": dense_flops / (asm_ms * 1e-3) / 1e12,
            "algorithmic_note": "SURVEY.md 8(d) dense count 4mn^3 + m(m+1)n^2 (what the reference's formulation executes); "
                                "algorithmic_speedup is the saving of the assembly form, reported separately from frac",
            "traffic": traffic["bytes"] if traffic else None,
            "traffic_source": traffic["source"] if traffic else "no ncu --set full capture of this form / shape",
        },
        "e2e": {"value": e2e_ms, "unit": UNIT, "h2d_bytes_per_step": 8 * m / e2e_its,
                "d2h_bytes_per_step": 8 * m / e2e_its + 8 * (2 * (n // 2 + 2) + 8) * 2 + 4 * 8 + 4,
                "device_step_ms": e2e_step_ms, "wall_ms": e2e_wall * 1e3,
                "note": "CONEX_Maximize warm-start solve of K steps from host b to host y; per-step D2H = Lanczos "
                        "coefficients + scalars. The operator itself is generated in place in library-owned HBM "
                        "(CONEXB200_NewDenseLMIConstraintStorage) once per program: setup_s; it is not re-sent per step"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "setup_s": setup_s, "first_solve_wall_s": wall_cold,
        "final": {"by": log[-1]["by"], "cx": log[-1]["cx"], "mu": log[-1]["mu"]},
    }
    if world == 1 and steps >= 3:
        rate = measure_h2d_rate(torch)
        if rate:
            line["operator_setup"] = {
                "in_this_run_s": setup_s, "how": "generated in place in library-owned HBM (CONEXB200_NewDenseLMIConstraintStorage)",
                "h2d_GBps_measured": rate, "h2d_sample_bytes": 1 << 30,
                "host_buffer_path_estimate_s": 8.0 * m * n * n / (rate * 1e9),
                "note": "one-time cost of CONEX_AddDenseLMIConstraint with HOST matrices at this shape = operator bytes / the "
                        "pinned H2D rate measured here (the operator is copied once per program, never per step)"}
    if has_shard:
        line["shard_assembly_ms"] = dict(zip(["local_k1_and_diagonal_block", "stall_waiting_for_peer_chunks",
                                              "off_diagonal_contractions", "allreduce_of_H"], shard),
                                         note="last timed assembly, CUDA events on the compute stream, max over ranks")
    if solve:
        line["solve"] = solve
        line["solve_ms"], line["solve_iterations"], line["solved"] = solve["solve_ms"], solve["solve_iterations"], solve["solved"]
    if cpu_leg:
        line["cpu_baseline"] = cpu_baseline(w, 2, 1, sample_key="cpu_small")
    return line


def compact(line):
    """The keys of a secondary workload's record that go inside the main JSON line."""
    if line is None or "error" in line:
        return line
    keep = ("value", "unit", "n_gpus", "steps", "warmup", "config", "phase_ms", "shard_assembly_ms", "solve_ms", "programs_per_s",
            "programs_solved", "step_tflops_fp64", "gpu_launches")
    out = {k: line[k] for k in keep if k in line}
    out["roofline"] = {k: line["roofline"][k] for k in ("bound", "achieved", "peak", "unit", "frac") if k in line["roofline"]}
    out["e2e"] = {k: line["e2e"][k] for k in ("value", "unit") if k in line["e2e"]}
    return out


def run_b200(args):
    proc = Process()
    if args.gemm_max_ktiles >= 0:
        proc.L.cxb_set_gemm_split_policy(args.gemm_max_ktiles)
    if args.gemm_config >= 0:
        proc.L.cxb_set_default_gemm_config(args.gemm_config)
    if args.gram_config >= -1:
        proc.L.cxb_set_gram_gemm_config(args.gram_config)
    w = workload_shape(args)
    outputs = {} if args.dump_outputs else None
    line = dense_bench(proc, args, w, args.steps, args.warmup, full_solve=not args.no_full_solve,
                       cpu_leg=not args.no_cpu_baseline and proc.rank == 0 and proc.world == 1, outputs=outputs)
    if args.workload == "c2" and not args.no_extra and not args.n and not args.m:
        # The other two shapes the north star quotes scaling on ride along in the same JSON line, so that the driver's
        # 1/2/4/8-GPU runs carry them: C5 (n = 1000, m = 20000; multi-GPU Cholesky on) and C3 (4096 small programs).
        # (a failure of a secondary block must not take the main line with it; every rank runs the same code on the
        # same shapes, so an exception is raised on all of them or on none)
        # The outputs of a block go into the dump only when the block has returned a result.
        c5_out = {} if outputs is not None else None
        try:
            c5w = workload_shape(argparse.Namespace(workload="c5", n=0, m=0, programs=0))
            c5 = compact(dense_bench(proc, args, c5w, 2, 1, full_solve=False, cpu_leg=False, outputs=c5_out))
            if c5 is not None and "error" not in c5:
                c5["note"] = "1 warm-up + 2 timed Newton steps whatever --steps / --warmup ask (a step is 1.3-14 s at this shape)"
                if outputs is not None:
                    outputs.update({"c5_" + k: v for k, v in c5_out.items()})
        except Exception as e:  # noqa: BLE001
            c5 = {"error": f"{type(e).__name__}: {e}"}
        c3_out = {} if outputs is not None else None
        try:
            c3w = workload_shape(argparse.Namespace(workload="c3", n=0, m=0, programs=0))
            c3 = compact(batched_bench(proc, args, c3w, args.steps, args.warmup, cpu_leg=False, outputs=c3_out))
            if outputs is not None:
                outputs.update({"c3_" + k: v for k, v in c3_out.items()})
        except Exception as e:  # noqa: BLE001
            c3 = {"error": f"{type(e).__name__}: {e}"}
        if line is not None:
            line["c5"] = c5
            line["c3"] = c3
    if line is not None:
        print(json.dumps(line))
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
    proc.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed Newton steps (c3: lock steps of the batch); the C5 block of the c2 line always times 2")
    ap.add_argument("--warmup", type=int, default=3, help="untimed Newton steps before them (at least 3 on the B200 arm)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS),
                    help="BASELINE.json configuration (c2 = MaxCut n=2000, the headline)")
    ap.add_argument("--size", dest="n", type=int, default=0, help="override the PSD order n")
    ap.add_argument("--constraints", dest="m", type=int, default=0, help="override the number of constraints m")
    ap.add_argument("--assembly-mode", type=int, default=0, help="0 auto, 1 classic (keep all W A_i W), 2 stream row panels, 3 symmetric form (packed L^T A_i L)")
    ap.add_argument("--programs", type=int, default=0, help="c3: number of programs in the batch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-full-solve", action="store_true", help="skip the default-configuration solve to termination")
    ap.add_argument("--no-extra", action="store_true", help="c2: skip the C5 and C3 blocks that ride along in the line")
    ap.add_argument("--cpu-size", type=int, default=0, help="override n = m of the CPU sample (testing)")
    ap.add_argument("--no-peer-memory", action="store_true",
                    help="N > 1 A/B: exchange the scaled matrices through ncclSend / ncclRecv instead of peer memory")
    ap.add_argument("--gemm-config", type=int, default=-1, help="A/B: cxb_set_default_gemm_config (tile configuration of the large GEMMs)")
    ap.add_argument("--gram-config", type=int, default=-2, help="A/B: cxb_set_gram_gemm_config (-1 = as the other large products)")
    ap.add_argument("--gemm-max-ktiles", type=int, default=-1, help="A/B: cxb_set_gemm_split_policy")
    ap.add_argument("--small-psd-mma", type=int, default=-1, help="c3 A/B: cxb_set_small_psd_mma (2 default, 1, 0)")
    ap.add_argument("--small-cone-threads", type=int, default=0, help="c3 A/B: cxb_set_small_cone_threads (32/64/128)")
    ap.add_argument("--small-fused-launches", type=int, default=-1, help="c3 A/B: cxb_set_small_fused_launches (0/1)")
    ap.add_argument("--small-team-mode", type=int, default=-1, help="c3 A/B: cxb_set_small_team_mode (1 default, 0)")
    ap.add_argument("--replicated-cholesky", action="store_true",
                    help="N > 1: factor the Schur complement on every rank instead of across the ranks")
    ap.add_argument("--cholesky-block", type=int, default=0, help="N > 1: block-column width (<= 512)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="B200 arm: after the timed steps, write what the timed solve returned (y, the iteration log; "
                         "c2 also the C5 / C3 blocks as c5_*, c3_*) as DIR/<name>.npy in float64")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the B200 arm")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif WORKLOADS[args.workload]["kind"] == "batched":
        run_b200_batched(args)
    elif WORKLOADS[args.workload]["kind"].endswith("_entries"):
        run_b200_structured(args)
    elif WORKLOADS[args.workload]["kind"] == "arrow":
        run_b200_sparse(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
