#!/usr/bin/env python
"""Batched solves of long MPC horizons, whose KKT systems do not fit in shared memory
(conex_b200.workloads.mpc_problem at 32 stages of 6 variables, m = 192; per stage an LP block of 12 rows and a
second-order cone of order 6, per pair of adjacent stages a dense LMI of order 8 and, in "eq", an equality block of 4
rows; every cone on its own variables):
  "eq"   : 32 stages with the equality blocks, KKT order N = 316: the blocked regularised LDL^T;
  "noeq" : 32 stages without them (eq_rows = 0), N = 192: the blocked Cholesky.

Per workload, `--programs` programs in one batch:
  * lock step: one solve of W + K Newton steps without final centering, CUDA events around each lock step
    (BatchProgram::step_milliseconds), mean of the K timed steps; kernel launches per lock step;
  * factorisation alone: cxb_small_ldlt / cxb_small_potrf on `--programs` copies of the cold-start KKT systems of
    the first 32 programs of the batch (CONEXB200_AssembleNewtonSystem), CUDA events around each of `--reps`
    launches (the Cholesky's input is restored between launches, outside the events); the solves
    (cxb_small_ldlt_solve / cxb_small_potrs) on the factors the same way. FLOP/s: N^3 / 3 per program over the
    kernel time; bytes: the lower triangle read once and written once;
  * whole solve: the default configuration from a cold start to termination (device ms, programs/s, iterations);
  * CONEX_Maximize, one program at a time, on the first `--sample` programs, host clock per call, extrapolated to the
    batch.
And, kernel level only, the blocked kernels against the shared-memory kernels at N = 76 and N = 168 (both fit in shared
memory, so cxb_small_potrf / cxb_small_ldlt take the shared-memory kernels there).

  python tools/batch_long_horizon_bench.py [--programs 4096] [--steps 10] [--warmup 3] [--reps 10] [--sample 32]
                                           [--out FILE]

Prints one JSON document (and writes it to FILE). Needs a GPU and the built library (__graft_entry__.build()).
"""
import argparse
import ctypes as C
import json
import multiprocessing
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from conex_b200.binding import Batch, product  # noqa: E402
from conex_b200.workloads import add_cones, mpc_problem  # noqa: E402

STAGES = 32
WORKLOADS = {"eq": dict(stages=STAGES), "noeq": dict(stages=STAGES, eq_rows=0)}
vp = C.c_void_p


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm,clocks.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        pl, mx, clk = [x.strip() for x in q.stdout.strip().split(",")[:3]]
        out.update(power_limit_w=float(pl), max_sm_mhz=float(mx), sm_mhz_now=float(clk))
    except (OSError, ValueError, subprocess.TimeoutExpired):
        out.update(power_limit_w=None, max_sm_mhz=None, sm_mhz_now=None)
    return out


def cublas_dgemm_tflops():
    """cuBLAS DGEMM 8192^3 through torch, best of 5: the FP64 denominator of bench.py."""
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


def _generate(args):
    seed, kw = args
    return mpc_problem(seed, **kw)


def build(dev, kw, count):
    with multiprocessing.get_context("fork").Pool(min(32, os.cpu_count() or 1)) as pool:
        problems = pool.map(_generate, [(2000 + p, kw) for p in range(count)], chunksize=16)
    programs, bs = [], []
    for cones, _, b in problems:
        P = dev.program(b.size)
        add_cones(P, cones)
        programs.append(P)
        bs.append(b)
    return programs, np.stack(bs)


def events_ms(fn, reps, before=None):
    """CUDA events around each of `reps` calls of fn (before() runs outside the events); mean and min in ms."""
    import torch
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        if before is not None:
            before()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return float(np.mean(times)), float(np.min(times))


class Kernels:
    """The four batched KKT entry points on `batch` column-major N x N matrices held by torch."""

    def __init__(self, lib):
        self.lib = lib
        for name in ("cxb_small_potrf", "cxb_small_potrf_blocked"):
            getattr(lib, name).argtypes = [vp, C.c_int, C.c_int, vp, C.c_long, C.c_long, vp, vp]
        for name in ("cxb_small_ldlt", "cxb_small_ldlt_blocked"):
            getattr(lib, name).argtypes = [vp, C.c_int, C.c_int, vp, C.c_long, C.c_long, vp, C.c_long, C.c_long, vp,
                                           C.c_long, vp, C.c_long, vp, vp]
        lib.cxb_small_potrs.argtypes = [vp, C.c_int, C.c_int, vp, C.c_long, C.c_long, vp, C.c_long, vp]
        lib.cxb_small_ldlt_solve.argtypes = [vp, C.c_int, C.c_int, vp, C.c_long, C.c_long, vp, C.c_long, vp, C.c_long,
                                             vp, C.c_long, vp]

    def setup(self, K):
        """K: torch (batch, N, N) float64 on the device, symmetric."""
        import torch
        self.B, self.N = K.shape[0], K.shape[1]
        self.K = K.contiguous()
        self.H = self.K.clone()
        self.L = torch.zeros_like(self.K)
        self.perm = torch.zeros((self.B, self.N), dtype=torch.int32, device="cuda")
        self.signs = torch.zeros((self.B, self.N), dtype=torch.float64, device="cuda")
        self.info = torch.zeros(self.B, dtype=torch.int32, device="cuda")
        self.x = torch.ones((self.B, self.N), dtype=torch.float64, device="cuda")

    def potrf(self, blocked=False):
        f = self.lib.cxb_small_potrf_blocked if blocked else self.lib.cxb_small_potrf
        N = self.N
        assert f(None, self.B, N, self.H.data_ptr(), N, N * N, self.info.data_ptr(), None) == 0

    def ldlt(self, blocked=False):
        f = self.lib.cxb_small_ldlt_blocked if blocked else self.lib.cxb_small_ldlt
        N = self.N
        assert f(None, self.B, N, self.K.data_ptr(), N, N * N, self.L.data_ptr(), N, N * N, self.perm.data_ptr(), N,
                 self.signs.data_ptr(), N, self.info.data_ptr(), None) == 0

    def potrs(self):
        N = self.N
        assert self.lib.cxb_small_potrs(None, self.B, N, self.H.data_ptr(), N, N * N, self.x.data_ptr(), N,
                                        None) == 0

    def ldlt_solve(self):
        N = self.N
        assert self.lib.cxb_small_ldlt_solve(None, self.B, N, self.L.data_ptr(), N, N * N, self.perm.data_ptr(), N,
                                             self.signs.data_ptr(), N, self.x.data_ptr(), N, None) == 0

    def restore(self):
        self.H.copy_(self.K)

    def time_factor(self, ldlt, reps, blocked=False):
        if ldlt:
            return events_ms(lambda: self.ldlt(blocked), reps)
        return events_ms(lambda: self.potrf(blocked), reps, before=self.restore)

    def time_solve(self, ldlt, reps):
        self.restore()
        if ldlt:
            self.ldlt()
            return events_ms(self.ldlt_solve, reps)
        self.potrf()
        return events_ms(self.potrs, reps)


def factor_metrics(N, B, ms, dgemm):
    flops = B * N ** 3 / 3.0
    bytes_ = 2.0 * B * N * (N + 1) / 2 * 8  # lower triangle read once, written once
    tflops = flops / (ms * 1e-3) / 1e12
    return {"flops": flops, "tflops": tflops, "fraction_of_cublas_dgemm": tflops / dgemm,
            "gbytes_per_s_lower_triangle_once": bytes_ / (ms * 1e-3) / 1e9}


def measure_workload(dev, name, kw, args, kern, dgemm):
    import torch
    lib = dev.lib
    lib.CONEXB200_LaunchCount.restype = C.c_long
    t0 = time.perf_counter()
    programs, b = build(dev, kw, args.programs)
    out = {"setup_s": time.perf_counter() - t0, "m": int(b.shape[1]), "kkt_order": int(programs[0].kkt_size())}
    N = out["kkt_order"]
    ldlt = name == "eq"
    # the factorisation and the solves alone, on copies of the first 32 programs' cold-start KKT systems
    sample = []
    for P in programs[:32]:
        H = P.newton_system(coldstart=True)[0]
        sample.append(H + np.tril(H, -1).T)
    K = torch.from_numpy(np.stack(sample)).cuda()  # symmetric: row- and column-major alike
    K = K.repeat((args.programs + 31) // 32, 1, 1)[:args.programs].contiguous()
    kern.setup(K)
    f_mean, f_min = kern.time_factor(ldlt, args.reps)
    s_mean, s_min = kern.time_solve(ldlt, args.reps)
    assert int((kern.info != 0).sum()) == 0 or ldlt, "cold-start Cholesky failed"
    out["factorisation"] = {"kernel": "cxb_small_ldlt (blocked LDL^T)" if ldlt else "cxb_small_potrf (blocked)",
                            "ms_mean": f_mean, "ms_min": f_min, **factor_metrics(N, args.programs, f_mean, dgemm)}
    out["solve"] = {"kernel": "cxb_small_ldlt_solve" if ldlt else "cxb_small_potrs", "ms_mean": s_mean,
                    "ms_min": s_min}
    del kern.K, kern.H, kern.L, K
    torch.cuda.empty_cache()
    # lock steps and the whole solve
    batch = Batch(dev, programs)
    cfg = dev.default_config(max_iterations=args.warmup + args.steps, final_centering_steps=0, inv_sqrt_mu_max=1e12)
    launches0 = lib.CONEXB200_LaunchCount()
    batch.maximize(b, cfg)
    launches = lib.CONEXB200_LaunchCount() - launches0
    step_ms = batch.step_milliseconds()
    out["lock_step"] = {"ms_mean": float(step_ms[args.warmup:].mean()),
                        "ms_each": [round(float(v), 4) for v in step_ms[args.warmup:]],
                        "launches": launches / len(step_ms)}
    out["lock_step"]["factorisation_share"] = f_mean / out["lock_step"]["ms_mean"]
    out["lock_step"]["two_solves_share"] = 2 * s_mean / out["lock_step"]["ms_mean"]
    t0 = time.perf_counter()
    solved, y = batch.maximize(b, dev.default_config())
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    its = batch.results()[0]
    ms = batch.milliseconds()
    out["solve_default"] = {"ms": ms, "wall_ms": 1e3 * wall, "programs_per_s": args.programs / (ms * 1e-3),
                            "lock_steps": int(len(batch.step_milliseconds())), "solved": int(np.sum(solved)),
                            "iterations_mean": float(its.mean()), "iterations_min": int(its.min()),
                            "iterations_max": int(its.max())}
    # CONEX_Maximize one program at a time
    times, yd = [], []
    for p in range(args.sample):
        t0 = time.perf_counter()
        s1, y1 = programs[p].maximize(b[p], dev.default_config())
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
        yd.append(np.abs(y1 - y[p]).max() / max(1.0, np.abs(y1).max()))
    per = float(np.mean(times))
    out["conex_maximize"] = {"sample": args.sample, "ms_per_program_mean": 1e3 * per,
                             "ms_per_program_median": 1e3 * float(np.median(times)),
                             "extrapolated_batch_ms": 1e3 * per * args.programs,
                             "batch_speedup": 1e3 * per * args.programs / ms,
                             "max_rel_y_difference_to_batch": float(max(yd))}
    del batch, programs
    return out


def measure_small(kern, args, dgemm):
    """Blocked against shared-memory kernels where both run."""
    import torch
    rng = np.random.Generator(np.random.PCG64(5))
    out = {}
    for N in (76, 168):
        rows = 28 if N == 76 else 64
        m = N - rows
        R = rng.uniform(-1, 1, size=(32, m, m + 2))
        Hs = R @ R.transpose(0, 2, 1) + 0.5 * np.eye(m)
        A = rng.uniform(-1, 1, size=(32, rows, m))
        K = np.zeros((32, N, N))
        K[:, :m, :m] = Hs
        K[:, m:, :m] = A
        K[:, :m, m:] = A.transpose(0, 2, 1)
        S = rng.uniform(-1, 1, size=(32, N, N + 2))
        P = S @ S.transpose(0, 2, 1) / N + np.eye(N)
        for kind, mats, ldlt in (("ldlt", K, True), ("potrf", P, False)):
            T = torch.from_numpy(mats).cuda().repeat(args.programs // 32, 1, 1).contiguous()
            kern.setup(T)
            shared = kern.time_factor(ldlt, args.reps, blocked=False)[0]
            blocked = kern.time_factor(ldlt, args.reps, blocked=True)[0]
            out[f"{kind}_N{N}"] = {"shared_ms": shared, "blocked_ms": blocked, "blocked_over_shared": blocked / shared,
                                   "faster": "blocked" if blocked < shared else "shared",
                                   "blocked_tflops": factor_metrics(N, args.programs, blocked, dgemm)["tflops"],
                                   "shared_tflops": factor_metrics(N, args.programs, shared, dgemm)["tflops"]}
            del kern.K, kern.H, kern.L, T
            torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--programs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--sample", type=int, default=32)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("batch_long_horizon_bench.py needs a GPU")
    dev = product()
    kern = Kernels(dev.lib)
    result = {"card": card(), "programs": args.programs, "stages": STAGES, "stage_variables": 6,
              "steps": args.steps, "warmup": args.warmup, "reps": args.reps}
    result["cublas_dgemm_8192_tflops"] = dgemm = cublas_dgemm_tflops()
    result["small_n_kernels"] = measure_small(kern, args, dgemm)
    for name, kw in WORKLOADS.items():
        result[name] = measure_workload(dev, name, kw, args, kern, dgemm)
    result["card_after"] = card()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
