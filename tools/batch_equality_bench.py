#!/usr/bin/env python
"""Batched solves with and without equality constraints on the C3 shape (4096 programs; 3 dense LMI blocks 20 x 20,
2 second-order cones of order 10, one LP block of 40 rows; m = 40): the plain batch (KKT order 40, Cholesky,
cxb_small_potrf / cxb_small_potrs) against the same programs with one equality block of 8 rows on all variables
(KKT order 48, regularised LDL^T, cxb_small_ldlt / cxb_small_ldlt_solve).

The two batches are measured alternately, `--rounds` times each, in one process:
  * lock step: one solve of W + K Newton steps without final centering (every program takes a full step in each),
    CUDA events around each lock step (BatchProgram::step_milliseconds), mean of the K timed steps;
  * whole solve: the default configuration from a cold start to termination (device ms, programs/s, iterations).
Then the two factorisations alone at N = 48 (and Cholesky at N = 40, the order of the plain batch), CUDA events
around `--launches` launches on 4096 matrices each; every Cholesky launch gets its own copy of the input (the
factorisation is in place), the LDL^T leaves its input as it is.

  python tools/batch_equality_bench.py [--programs 4096] [--steps 20] [--warmup 5] [--rounds 3] [--out FILE]

Prints one JSON document (and writes it to FILE). Needs a GPU and the built library (__graft_entry__.build()).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from conex_b200.binding import Batch, product  # noqa: E402
from conex_b200.workloads import add_cones, small_multicone_equality_problem, small_multicone_problem  # noqa: E402

C3 = dict(m=40, psd_blocks=3, psd_order=20, soc_cones=2, soc_order=10, lp_rows=40)
EQ_ROWS = 8


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        pl, clk = [x.strip() for x in q.stdout.strip().split(",")[:2]]
        out.update(power_limit_w=float(pl), max_sm_mhz=float(clk))
    except (OSError, ValueError, subprocess.TimeoutExpired):
        out.update(power_limit_w=None, max_sm_mhz=None)
    return out


def build_batch(dev, count, equalities):
    programs, bs = [], []
    for p in range(count):
        if equalities:
            cones, b = small_multicone_equality_problem(1000 + p, equalities=((EQ_ROWS, None, None),), **C3)
        else:
            cones, b = small_multicone_problem(1000 + p, **C3)
        P = dev.program(C3["m"])
        add_cones(P, cones)
        programs.append(P)
        bs.append(b)
    return Batch(dev, programs), np.stack(bs)


def measure_batch(dev, batch, b, steps, warmup):
    import torch
    cfg = dev.default_config(max_iterations=warmup + steps, final_centering_steps=0, inv_sqrt_mu_max=1e12)
    batch.maximize(b, cfg)
    step_ms = batch.step_milliseconds()
    assert len(step_ms) == warmup + steps, len(step_ms)
    t0 = time.perf_counter()
    solved, _ = batch.maximize(b, dev.default_config())
    torch.cuda.synchronize()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    its = batch.results()[0]
    solve_ms = batch.milliseconds()
    return {"lock_step_ms": float(step_ms[warmup:].mean()), "lock_step_ms_each": [round(float(v), 4) for v in
                                                                                   step_ms[warmup:]],
            "solve_ms": solve_ms, "solve_wall_ms": wall_ms, "programs_per_s": len(b) / (solve_ms * 1e-3),
            "lock_steps": int(len(batch.step_milliseconds())), "iterations_mean": float(its.mean()),
            "iterations_min": int(its.min()), "iterations_max": int(its.max()), "solved": int(solved.sum())}


def kkt_batch(rng, count, m, rows):
    N = m + rows
    K = np.zeros((count, N, N))
    R = rng.uniform(-1.0, 1.0, size=(count, m, m + 2))
    K[:, :m, :m] = R @ R.transpose(0, 2, 1) + 0.5 * np.eye(m)
    if rows:
        A = rng.uniform(-1.0, 1.0, size=(count, rows, m))
        K[:, m:, :m] = A
        K[:, :m, m:] = A.transpose(0, 2, 1)
    return K


def kernel_times(lib, count, launches):
    """ms per launch of cxb_small_potrf (N = 40, 48), cxb_small_ldlt (N = 48) and their solves, CUDA events."""
    import torch
    vp = C.c_void_p
    lib.cxb_small_potrf.argtypes = [vp, C.c_int, C.c_int, vp, C.c_long, C.c_long, vp, vp]
    lib.cxb_small_potrs.argtypes = [vp, C.c_int, C.c_int, vp, C.c_long, C.c_long, vp, C.c_long, vp]
    lib.cxb_small_ldlt.argtypes = [vp, C.c_int, C.c_int, vp, C.c_long, C.c_long, vp, C.c_long, C.c_long, vp, C.c_long,
                                   vp, C.c_long, vp, vp]
    lib.cxb_small_ldlt_solve.argtypes = [vp, C.c_int, C.c_int, vp, C.c_long, C.c_long, vp, C.c_long, vp, C.c_long, vp,
                                         C.c_long, vp]
    rng = np.random.Generator(np.random.PCG64(7))
    out = {}

    def timed(fn, setup=None):
        for i in range(3):  # warm-up
            if setup:
                setup(i)
            fn(i)
        torch.cuda.synchronize()
        total = 0.0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for i in range(launches):
            if setup:
                setup(i)
            e0.record()
            fn(i)
            e1.record()
            e1.synchronize()
            total += e0.elapsed_time(e1)
        return total / launches

    def col_major(K):
        return torch.from_numpy(np.ascontiguousarray(K.transpose(0, 2, 1)).ravel()).cuda()

    for N in (40, 48):
        src = col_major(kkt_batch(rng, count, N, 0))
        work = torch.empty_like(src)
        info = torch.zeros(count, dtype=torch.int32, device="cuda")

        def potrf(i):
            assert lib.cxb_small_potrf(None, count, N, work.data_ptr(), N, N * N, info.data_ptr(), None) == 0

        out[f"potrf_N{N}_ms"] = timed(potrf, setup=lambda i: work.copy_(src))
        assert int(info.abs().max()) == 0
        rhs = torch.from_numpy(rng.uniform(-1, 1, size=count * N)).cuda()
        x = torch.empty_like(rhs)
        out[f"potrs_N{N}_ms"] = timed(lambda i: lib.cxb_small_potrs(None, count, N, work.data_ptr(), N, N * N,
                                                                    x.data_ptr(), N, None),
                                      setup=lambda i: x.copy_(rhs))
    m, rows = 40, 8
    N = m + rows
    K = col_major(kkt_batch(rng, count, m, rows))
    L = torch.zeros_like(K)
    perm = torch.zeros(count * N, dtype=torch.int32, device="cuda")
    signs = torch.zeros(count * N, dtype=torch.float64, device="cuda")
    info = torch.zeros(count, dtype=torch.int32, device="cuda")
    rhs = torch.from_numpy(rng.uniform(-1, 1, size=count * N)).cuda()
    x = torch.empty_like(rhs)

    def ldlt(i):
        assert lib.cxb_small_ldlt(None, count, N, K.data_ptr(), N, N * N, L.data_ptr(), N, N * N, perm.data_ptr(), N,
                                  signs.data_ptr(), N, info.data_ptr(), None) == 0

    out["ldlt_N48_ms"] = timed(ldlt)
    assert int(info.abs().max()) == 0
    out["ldlt_solve_N48_ms"] = timed(lambda i: lib.cxb_small_ldlt_solve(None, count, N, L.data_ptr(), N, N * N,
                                                                        perm.data_ptr(), N, signs.data_ptr(), N,
                                                                        x.data_ptr(), N, None),
                                      setup=lambda i: x.copy_(rhs))
    out.update(programs=count, launches=launches)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--programs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("batch_equality_bench.py needs a GPU")
    dev = product()
    result = {"card": card(), "shape": dict(C3, programs=args.programs, equality_rows=EQ_ROWS),
              "steps": args.steps, "warmup": args.warmup}
    t0 = time.perf_counter()
    batches = {"plain": build_batch(dev, args.programs, False), "equality": build_batch(dev, args.programs, True)}
    result["setup_s"] = time.perf_counter() - t0
    runs = {"plain": [], "equality": []}
    for _ in range(args.rounds):
        for name in ("plain", "equality"):
            batch, b = batches[name]
            runs[name].append(measure_batch(dev, batch, b, args.steps, args.warmup))
    for name, rs in runs.items():
        step = [r["lock_step_ms"] for r in rs]
        result[name] = {"lock_step_ms_median": float(np.median(step)), "lock_step_ms_min": float(min(step)),
                        "lock_step_ms_max": float(max(step)),
                        "solve_ms_median": float(np.median([r["solve_ms"] for r in rs])),
                        "programs_per_s_median": float(np.median([r["programs_per_s"] for r in rs])),
                        "rounds": rs}
    result["lock_step_ratio_equality_over_plain"] = (result["equality"]["lock_step_ms_median"] /
                                                     result["plain"]["lock_step_ms_median"])
    del batches
    result["kernels"] = kernel_times(dev.lib, args.programs, args.launches)
    result["card_after"] = card()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
