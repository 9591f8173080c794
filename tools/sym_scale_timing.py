#!/usr/bin/env python
"""Times K1 of the symmetric Schur form alone: cxb_schur_dense_lmi_sym_scale (Cholesky of W, the packed L^T A_i L of
every constraint matrix, L^T C L and I) at n = 2000, on one panel of the C2 step (33 matrices, m = 32) and on the
whole scale phase of C2 (m = 2000, panel 33 as the dense LMI constraint picks it). CUDA events around each call, best
and median of --reps calls after one warm-up call; operands of 1 GB (panel) and 64 GB (whole phase) are far larger
than L2.

Executed TFLOP/s use the K1 flop count of the build being timed, --k1-n3 * (m + 1) * n^3: 1.0 for this tree (Y_i =
tril-half(A_i) L, then L^T Y_i + Y_i^T L), 4/3 for builds that form A_i L and L^T (A_i L). Only the exported entry
point is called, so the same script times any build of the library. One JSON line per case, also appended to --out.

  python tools/sym_scale_timing.py --label pr --out profiles/r03_sym_scale_timing.jsonl
  python tools/sym_scale_timing.py --label parent --k1-n3 1.3333333333333333 --out ...
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import conex_b200.binding as dev  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=2000)
    ap.add_argument("--panel", type=int, default=33)
    ap.add_argument("--cases", default="panel,phase", help="panel: m = panel - 1 (one launch pair); phase: m = 2000")
    ap.add_argument("--m-phase", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--k1-n3", type=float, default=1.0, help="executed K1 flops per matrix / n^3 of this build")
    ap.add_argument("--label", default="")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sym_scale_timing.py needs a CUDA device")

    L = dev.product().lib
    vp = C.c_void_p
    L.cxb_packed_symmetric_size.restype = C.c_size_t
    L.cxb_packed_symmetric_size.argtypes = [C.c_int]
    L.cxb_schur_dense_lmi_sym_scale.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp, C.c_int, vp, vp]
    n, panel = args.n, args.panel
    nn = n * n
    kp = L.cxb_packed_symmetric_size(n)
    gen = torch.Generator(device="cuda").manual_seed(7)
    R = torch.rand((n, n), dtype=torch.float64, device="cuda", generator=gen)
    W = (R @ R.T / n + torch.eye(n, dtype=torch.float64, device="cuda")).contiguous()
    dT = torch.empty(panel * nn, dtype=torch.float64, device="cuda")
    dL = torch.empty(nn, dtype=torch.float64, device="cuda")
    info = torch.zeros(2, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream()
    card = gpu_info()
    for case in args.cases.split(","):
        m = panel - 1 if case == "panel" else args.m_phase
        A = torch.rand((m + 1) * nn, dtype=torch.float64, device="cuda", generator=gen).sub_(0.5)
        X = torch.empty((m + 2) * kp, dtype=torch.float64, device="cuda")

        def call():
            rc = L.cxb_schur_dense_lmi_sym_scale(vp(stream.cuda_stream), n, m, dev.ptr(A), dev.ptr(W), dev.ptr(X),
                                                 dev.ptr(dT), panel, dev.ptr(dL), dev.ptr(info))
            assert rc == 0, rc

        call()
        torch.cuda.synchronize()
        assert int(info[0]) == 0
        ts = []
        for _ in range(args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            call()
            e1.record(stream)
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / 1e3)
        flops = args.k1_n3 * (m + 1) * float(n) ** 3
        line = dict(kernel="cxb_schur_dense_lmi_sym_scale", label=args.label, case=case, n=n, m=m, panel=panel,
                    reps=args.reps, best_s=min(ts), median_s=float(np.median(ts)), k1_n3=args.k1_n3,
                    executed_flops=flops, executed_TFLOPs=flops / min(ts) / 1e12, gpu=card)
        print(json.dumps(line), flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(json.dumps(line) + "\n")
        del A, X
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
