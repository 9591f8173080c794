#!/usr/bin/env python
"""Warm starts of a batch across a sequence of nearby instances, on the C3 shape (4096 programs; 3 dense LMI blocks
20 x 20, 2 second-order cones of order 10, one LP block of 40 rows; m = 40) — the loop of a model-predictive
controller or a parameter sweep: change the data in place, solve again from the previous iterate.

Two batches are built from the same programs. For each eps in --eps, both are first reset to the original data and
solved from a cold start; then `--ticks` times:
  * the affine term of every cone of every program is perturbed, C <- C + eps sym(U[-1,1]) (LMI), c <- c + eps U[-1,1]
    (LP, second-order), with CONEXB200_BatchUpdateConstraintData on both batches (the same data);
  * batch "warm" is solved with initialization_mode = 1, batch "cold" from a cold start.
Per eps: the update time of one batch (host clock around the update calls, which end in a synchronise), the lock
steps, device ms (CUDA events, BatchProgram::milliseconds) and programs/s of the warm and of the cold solves, and the
largest |y_warm - y_cold| over the programs both solved.

  python tools/batch_warmstart_bench.py [--programs 4096] [--ticks 5] [--eps 1e-3 1e-2 1e-1] [--out FILE]

Prints one JSON document (and writes it to FILE). Needs a GPU and the built library (__graft_entry__.build()).
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

from batch_equality_bench import C3, card  # noqa: E402
from conex_b200.binding import Batch, product  # noqa: E402
from conex_b200.workloads import add_cones, small_multicone_problem  # noqa: E402


def affine_columns(cones):
    """Per constraint: (rows, base affine terms of every program as (count, rows, 1), is_lmi)."""
    out = []
    for k, (kind, _, _) in enumerate(cones[0]):
        base = np.stack([np.asarray(cs[k][2], dtype=np.float64).ravel(order="F") for cs in cones])
        out.append((base.shape[1], base[:, :, None], kind == "psd"))
    return out


def perturbation(rng, rows, count, is_lmi, eps):
    noise = rng.uniform(-1.0, 1.0, size=(count, rows, 1))
    if is_lmi:
        n = int(round(np.sqrt(rows)))
        N = noise.reshape(count, n, n)  # any fixed layout: the result is symmetrised
        noise = (0.5 * (N + N.transpose(0, 2, 1))).reshape(count, rows, 1)
    return eps * noise


def solve(dev, batch, b, warm):
    cfg = dev.default_config(initialization_mode=1 if warm else 0)
    solved, y = batch.maximize(b, cfg)
    return {"solved": solved, "y": y, "ms": batch.milliseconds(), "lock_steps": len(batch.step_milliseconds()),
            "iterations_mean": float(batch.results()[0].mean())}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--programs", type=int, default=4096)
    ap.add_argument("--ticks", type=int, default=5)
    ap.add_argument("--eps", type=float, nargs="+", default=[1e-3, 1e-2, 1e-1])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("batch_warmstart_bench.py needs a GPU")
    dev = product()
    B = args.programs
    result = {"card": card(), "shape": dict(C3, programs=B), "ticks": args.ticks}
    t0 = time.perf_counter()
    problems = [small_multicone_problem(1000 + p, **C3) for p in range(B)]
    programs = []
    for cones, _ in problems:
        P = dev.program(C3["m"])
        add_cones(P, cones)
        programs.append(P)
    batches = {"warm": Batch(dev, programs), "cold": Batch(dev, programs)}
    del programs
    b = np.stack([pb for _, pb in problems])
    columns = affine_columns([cones for cones, _ in problems])
    m = C3["m"]
    result["setup_s"] = time.perf_counter() - t0
    rng = np.random.Generator(np.random.PCG64(7))
    result["runs"] = []
    for eps in args.eps:
        current = [base.copy() for _, base, _ in columns]
        for batch in batches.values():
            for k, data in enumerate(current):
                batch.update(k, m, data)
        first = {name: solve(dev, batch, b, False) for name, batch in batches.items()}
        ticks = []
        for _ in range(args.ticks):
            for k, (rows, _, is_lmi) in enumerate(columns):
                current[k] = current[k] + perturbation(rng, rows, B, is_lmi, eps)
            t = time.perf_counter()
            for k, data in enumerate(current):
                batches["warm"].update(k, m, data)
            update_ms = 1e3 * (time.perf_counter() - t)
            for k, data in enumerate(current):
                batches["cold"].update(k, m, data)
            warm = solve(dev, batches["warm"], b, True)
            cold = solve(dev, batches["cold"], b, False)
            both = (warm["solved"] == 1) & (cold["solved"] == 1)
            dy = float(np.abs(warm["y"][both] - cold["y"][both]).max()) if both.any() else None
            ticks.append({"update_ms": update_ms, "max_abs_y_warm_minus_cold": dy,
                          **{f"{name}_{key}": (int(r["solved"].sum()) if key == "solved" else r[key])
                             for name, r in (("warm", warm), ("cold", cold))
                             for key in ("solved", "ms", "lock_steps", "iterations_mean")}})
        summary = {"eps": eps, "first_cold_ms": first["warm"]["ms"], "ticks": ticks}
        for name in ("warm", "cold"):
            ms = float(np.median([t[f"{name}_ms"] for t in ticks]))
            summary[name] = {"ms_median": ms, "programs_per_s_median": B / (ms * 1e-3),
                             "lock_steps_median": float(np.median([t[f"{name}_lock_steps"] for t in ticks])),
                             "iterations_mean": float(np.mean([t[f"{name}_iterations_mean"] for t in ticks])),
                             "solved_min": int(min(t[f"{name}_solved"] for t in ticks))}
        summary["update_ms_median"] = float(np.median([t["update_ms"] for t in ticks]))
        summary["max_abs_y_warm_minus_cold"] = max((t["max_abs_y_warm_minus_cold"] or 0.0) for t in ticks)
        summary["warm_over_cold_ms"] = summary["warm"]["ms_median"] / summary["cold"]["ms_median"]
        result["runs"].append(summary)
    result["card_after"] = card()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
