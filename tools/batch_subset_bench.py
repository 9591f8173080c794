#!/usr/bin/env python
"""Batched solves of MPC-shaped programs (conex_b200.workloads.mpc_problem: 8 stages of 6 variables, m = 48; per
stage an LP block of 12 rows and a second-order cone of order 6 on the stage's variables, per pair of adjacent stages
a dense LMI of order 8 and an equality block of 4 rows on the two stages' 12 variables; 23 cones, KKT order 76):
  (a) "subset": every cone on its own variables (the gather of y, the per-cone y source, the scatter-add of the
      Schur blocks);
  (b) "padded": the same programs with every cone zero-padded to all 48 variables — the only way to batch them
      without cones on variable subsets.

The two batches are measured alternately, `--rounds` times each, in one process:
  * lock step: one solve of W + K Newton steps without final centering, CUDA events around each lock step
    (BatchProgram::step_milliseconds), mean of the K timed steps; kernel launches per lock step
    (CONEXB200_LaunchCount);
  * whole solve: the default configuration from a cold start to termination (device ms, programs/s, iterations).
The largest |y_a - y_b| over the programs compares the answers of the two whole solves.

  python tools/batch_subset_bench.py [--programs 4096] [--steps 20] [--warmup 5] [--rounds 3] [--out FILE]

Prints one JSON document (and writes it to FILE). Needs a GPU and the built library (__graft_entry__.build()).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from conex_b200.binding import Batch, product  # noqa: E402
from conex_b200.workloads import add_cones, mpc_problem  # noqa: E402


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


def build_batches(dev, count):
    subset, padded, bs = [], [], []
    for p in range(count):
        cones, pad, b = mpc_problem(1000 + p)
        for target, cs in ((subset, cones), (padded, pad)):
            P = dev.program(b.size)
            add_cones(P, cs)
            target.append(P)
        bs.append(b)
    return {"subset": Batch(dev, subset), "padded": Batch(dev, padded)}, np.stack(bs)


def measure(dev, batch, b, steps, warmup):
    import torch
    lib = dev.lib
    lib.CONEXB200_LaunchCount.restype = ctypes.c_long
    cfg = dev.default_config(max_iterations=warmup + steps, final_centering_steps=0, inv_sqrt_mu_max=1e12)
    launches0 = lib.CONEXB200_LaunchCount()
    batch.maximize(b, cfg)
    launches = lib.CONEXB200_LaunchCount() - launches0
    step_ms = batch.step_milliseconds()
    assert len(step_ms) == warmup + steps, len(step_ms)
    t0 = time.perf_counter()
    solved, y = batch.maximize(b, dev.default_config())
    torch.cuda.synchronize()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    its = batch.results()[0]
    solve_ms = batch.milliseconds()
    return y, {"lock_step_ms": float(step_ms[warmup:].mean()),
               "lock_step_ms_each": [round(float(v), 4) for v in step_ms[warmup:]],
               "launches_per_lock_step": launches / (warmup + steps),
               "solve_ms": solve_ms, "solve_wall_ms": wall_ms, "programs_per_s": len(b) / (solve_ms * 1e-3),
               "lock_steps": int(len(batch.step_milliseconds())), "iterations_mean": float(its.mean()),
               "iterations_min": int(its.min()), "iterations_max": int(its.max()), "solved": int(solved.sum())}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--programs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("batch_subset_bench.py needs a GPU")
    dev = product()
    result = {"card": card(), "shape": dict(programs=args.programs, stages=8, stage_variables=6, m=48, cones=23,
                                            kkt_order=76, lp_rows=12, soc_order=6, lmi_order=8, equality_rows=4),
              "steps": args.steps, "warmup": args.warmup}
    t0 = time.perf_counter()
    batches, b = build_batches(dev, args.programs)
    result["setup_s"] = time.perf_counter() - t0
    runs = {"subset": [], "padded": []}
    answers = {}
    for _ in range(args.rounds):
        for name in ("subset", "padded"):
            y, r = measure(dev, batches[name], b, args.steps, args.warmup)
            runs[name].append(r)
            answers[name] = y
    for name, rs in runs.items():
        step = [r["lock_step_ms"] for r in rs]
        result[name] = {"lock_step_ms_median": float(np.median(step)), "lock_step_ms_min": float(min(step)),
                        "lock_step_ms_max": float(max(step)),
                        "solve_ms_median": float(np.median([r["solve_ms"] for r in rs])),
                        "programs_per_s_median": float(np.median([r["programs_per_s"] for r in rs])),
                        "iterations_mean": rs[-1]["iterations_mean"], "iterations_max": rs[-1]["iterations_max"],
                        "launches_per_lock_step": rs[-1]["launches_per_lock_step"], "rounds": rs}
    result["lock_step_ratio_subset_over_padded"] = (result["subset"]["lock_step_ms_median"] /
                                                    result["padded"]["lock_step_ms_median"])
    result["solve_ratio_subset_over_padded"] = (result["subset"]["solve_ms_median"] /
                                                result["padded"]["solve_ms_median"])
    result["added_launches_per_lock_step"] = (result["subset"]["launches_per_lock_step"] -
                                              result["padded"]["launches_per_lock_step"])
    result["max_abs_y_difference"] = float(np.abs(answers["subset"] - answers["padded"]).max())
    result["card_after"] = card()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
