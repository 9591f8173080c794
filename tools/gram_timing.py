#!/usr/bin/env python
"""Times K2 of the symmetric Schur form alone at the C2 shape (MaxCut n = m = 2000: X is K = kp(2000) = 2 162 688 by
m + 2 = 2002, 35 GB of FP64): cxb_schur_dense_lmi_sym_gram_ws with the slice workspace (the int8 emulated Gram,
slicing included), the slicing alone (cxb_gram_slices), and with a null workspace (the DMMA Gram). CUDA events around
--reps launches after one warm-up launch of each. X is random normal (the kernels' time does not depend on the
values). Prints and appends one JSON line per arm to --out: milliseconds per launch, and for the emulated Gram the int8
operations its tensor cores execute (every lower 128 x 64 tile, 36 slice products, K rounded up to the 32-byte k-step)
per second, beside the 4.5 POP/s dense INT8 figure of the B200 data sheet (a data-sheet number, not a measurement).

  python tools/gram_timing.py --out gram_timing.jsonl
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=2000)
    ap.add_argument("--m", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--label", default="")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    import torch
    import conex_b200.binding as devlib
    L = devlib.product().lib
    vp = C.c_void_p
    L.cxb_packed_symmetric_size.restype = C.c_size_t
    L.cxb_packed_symmetric_size.argtypes = [C.c_int]
    L.cxb_schur_dense_lmi_sym_gram_workspace.restype = C.c_size_t
    L.cxb_schur_dense_lmi_sym_gram_workspace.argtypes = [C.c_int, C.c_int]
    L.cxb_schur_dense_lmi_sym_gram_ws.argtypes = [vp, C.c_int, C.c_int, vp, vp, C.c_long, vp, C.c_size_t]
    L.cxb_gram_slices.argtypes = [vp, C.c_int, C.c_long, vp, C.c_long, vp]
    n, m = args.n, args.m
    kp = L.cxb_packed_symmetric_size(n)
    M, N = m + 2, m + 1
    ldh = (M + 1) & ~1
    gen = torch.Generator(device="cuda").manual_seed(1)
    X = torch.empty(M * kp, dtype=torch.float64, device="cuda")
    for j in range(M):
        X[j * kp:(j + 1) * kp].normal_(generator=gen)
    H = torch.zeros(ldh * N, dtype=torch.float64, device="cuda")
    need = L.cxb_schur_dense_lmi_sym_gram_workspace(n, m)
    work = torch.empty(need, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream()
    s = vp(stream.cuda_stream)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    arms = {
        "emulated_gram": lambda: L.cxb_schur_dense_lmi_sym_gram_ws(s, n, m, devlib.ptr(X), devlib.ptr(H), ldh,
                                                                   devlib.ptr(work), need),
        "slices_only": lambda: L.cxb_gram_slices(s, M, kp, devlib.ptr(X), kp, devlib.ptr(work)),
        "dmma_gram": lambda: L.cxb_schur_dense_lmi_sym_gram_ws(s, n, m, devlib.ptr(X), devlib.ptr(H), ldh, None, 0),
    }
    tiles_m = (M + 127) // 128
    tiles = sum(tiles_m - (tn * 64) // 128 for tn in range((N + 63) // 64))
    ksteps = (kp + 31) // 32
    int8_ops = tiles * 36 * 2 * 128 * 64 * 32 * ksteps
    with open(args.out, "a") as f:
        for name, fn in arms.items():
            assert fn() == 0, name
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(stream)
            for _ in range(args.reps):
                assert fn() == 0, name
            t1.record(stream)
            torch.cuda.synchronize()
            ms = t0.elapsed_time(t1) / args.reps
            line = dict(kernel=name, label=args.label, n=n, m=m, kp=kp, reps=args.reps, ms=ms, gpu=card)
            if name == "emulated_gram":
                line.update(int8_ops_executed=int8_ops, int8_pops_per_s=int8_ops / (ms * 1e-3) / 1e15,
                            datasheet_int8_dense_pops=4.5)
            print(json.dumps(line), flush=True)
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
