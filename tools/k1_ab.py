#!/usr/bin/env python
"""A/B of two prebuilt product libraries on the flagship line (MaxCut n = m = 2000, dense LMI path, one GPU), in one
session on one card, e.g. a build of the parent commit against a build of a change to K1 of the Schur assembly.

Before each run the chosen library is copied over conex_b200/lib/libconex_b200.so. The original is first copied to
libconex_b200.so.ab_original beside it and put back at the end; while an arm's library is in place, the file
libconex_b200.so.ab_swapped beside it names that arm. If the tool is killed before it restores the original, the marker
stays, and the next run of the tool restores the original before it does anything else. The runs, in this order:
  1. `bench.py --no-extra --no-cpu-baseline --no-full-solve --dump-outputs DIR`, alternating A, B, A, B, ... (--runs
     of each), so that drift of the card's clocks or of the host load falls on both arms alike;
  2. optionally tools/sym_scale_timing.py with each library (K1 alone; --timing);
  3. one full default `bench.py` with each library, A then B (--no-full-lines skips it).
Printed and written to OUT/summary.json: the card's name, power limit and maximum SM clock; per arm the median,
spread and every value (ms per Newton step) and phase_ms; the B / A ratio of the medians; the largest relative
differences of y and of every iteration-log column between the arms' dumps (same seeded inputs, different
rounding); the solve, c3 and c5 entries of the full lines. Every child process is waited for.

  python tools/k1_ab.py --a build/parent/libconex_b200.so --b conex_b200/lib/libconex_b200.so --out ab_out
"""
import argparse
import json
import os
import shutil
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "conex_b200", "lib", "libconex_b200.so")
ORIGINAL = LIB + ".ab_original"
MARKER = LIB + ".ab_swapped"
LOG_COLUMNS = ["inv_sqrt_mu", "mu", "d_2", "d_inf", "by", "cx", "kkt_error", "step_size"]


def card():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                          capture_output=True, text=True).stdout.strip()


def use(lib, arm):
    with open(MARKER, "w") as f:
        f.write(f"{LIB} is arm {arm}'s library ({lib}); the tree's own build is {ORIGINAL}\n")
    tmp = LIB + ".ab_tmp"
    shutil.copyfile(lib, tmp)
    os.replace(tmp, LIB)


def restore():
    """Puts the tree's own library back (also after an earlier run that was killed) and removes the marker."""
    if os.path.exists(ORIGINAL):
        tmp = LIB + ".ab_tmp"
        shutil.copyfile(ORIGINAL, tmp)
        os.replace(tmp, LIB)
        os.unlink(ORIGINAL)
    if os.path.exists(MARKER):
        os.unlink(MARKER)


def run(cmd, log):
    """Runs cmd to completion, output to `log`; returns the last JSON line it printed."""
    with open(log, "w") as f:
        p = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        f.write(p.stdout)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    if p.returncode != 0 or not lines:
        raise SystemExit(f"{' '.join(cmd)} failed (exit {p.returncode}), see {log}")
    return json.loads(lines[-1])


def rel_diff(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape:
        return None
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(a), 1e-300))) if a.size else 0.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--a", required=True, help="library of arm A (e.g. the parent commit)")
    ap.add_argument("--b", required=True, help="library of arm B")
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=3, help="bench runs per arm (alternating)")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--timing", action="store_true", help="also tools/sym_scale_timing.py with each library")
    ap.add_argument("--k1-n3", nargs=2, type=float, default=[4.0 / 3.0, 1.0], metavar=("A", "B"),
                    help="executed K1 flops per matrix / n^3 of each arm (for --timing)")
    ap.add_argument("--no-full-lines", action="store_true")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    out = os.path.abspath(args.out)
    arms = {"A": os.path.abspath(args.a), "B": os.path.abspath(args.b)}
    if os.path.exists(MARKER):
        print(f"restoring {LIB} left swapped by an earlier run: {open(MARKER).read().strip()}", flush=True)
        restore()
    shutil.copyfile(LIB, ORIGINAL + ".tmp")
    os.replace(ORIGINAL + ".tmp", ORIGINAL)
    summary = {"card": card(), "arms": arms}
    print(summary["card"], flush=True)
    try:
        lines = {"A": [], "B": []}
        for i in range(args.runs):
            for arm in ("A", "B"):
                use(arms[arm], arm)
                dump = os.path.join(out, f"dump_{arm}_{i}")
                line = run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(args.steps), "--warmup",
                            str(args.warmup), "--no-extra", "--no-cpu-baseline", "--no-full-solve", "--dump-outputs",
                            dump], os.path.join(out, f"bench_{arm}_{i}.log"))
                lines[arm].append(line)
                print(json.dumps({"arm": arm, "run": i, "value": line["value"], "phase_ms": line.get("phase_ms")}),
                      flush=True)
        for arm in ("A", "B"):
            v = [ln["value"] for ln in lines[arm]]
            summary[arm] = {"values": v, "median": float(np.median(v)), "min": min(v), "max": max(v),
                            "phase_ms": [ln.get("phase_ms") for ln in lines[arm]],
                            "roofline_frac": [ln.get("roofline", {}).get("frac") for ln in lines[arm]]}
        summary["median_ratio_B_over_A"] = summary["B"]["median"] / summary["A"]["median"]
        da, db = os.path.join(out, "dump_A_0"), os.path.join(out, "dump_B_0")
        ya, yb = np.load(os.path.join(da, "y.npy")), np.load(os.path.join(db, "y.npy"))
        la, lb = np.load(os.path.join(da, "iteration_log.npy")), np.load(os.path.join(db, "iteration_log.npy"))
        parity = {"y": rel_diff(ya, yb), "iterations": [len(la), len(lb)]}
        if la.shape == lb.shape:
            parity.update({c: rel_diff(la[:, j], lb[:, j]) for j, c in enumerate(LOG_COLUMNS)})
            # the first logged step whose by or cx differ by more than 1e-7 relative (None: none does)
            far = [i for i in range(len(la)) if max(rel_diff(la[i, 4], lb[i, 4]), rel_diff(la[i, 5], lb[i, 5])) > 1e-7]
            parity["first_step_by_cx_beyond_1e-7"] = far[0] if far else None
        parity["same_arm_runs_bit_identical"] = all(
            np.array_equal(np.load(os.path.join(out, f"dump_{arm}_0", "y.npy")),
                           np.load(os.path.join(out, f"dump_{arm}_{i}", "y.npy")))
            for arm in ("A", "B") for i in range(1, args.runs))
        summary["parity_max_rel_diff"] = parity
        if args.timing:
            path = os.path.join(out, "sym_scale_timing.jsonl")
            for arm, k1 in zip(("A", "B"), args.k1_n3):
                use(arms[arm], arm)
                run([sys.executable, os.path.join("tools", "sym_scale_timing.py"), "--label", arm, "--k1-n3", str(k1),
                     "--out", path], os.path.join(out, f"timing_{arm}.log"))
            summary["sym_scale_timing"] = [json.loads(ln) for ln in open(path)]
        if not args.no_full_lines:
            full = {}
            for arm in ("A", "B"):
                use(arms[arm], arm)
                line = run([sys.executable, "bench.py"], os.path.join(out, f"bench_full_{arm}.log"))
                full[arm] = {k: line.get(k) for k in ("value", "phase_ms", "solve_ms", "solve_iterations", "solved",
                                                       "c3", "c5")}
            summary["full_lines"] = full
    finally:
        restore()
        summary["card_after"] = card()
        with open(os.path.join(out, "summary.json"), "w") as f:
            json.dump(summary, f, indent=1)
    print(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
