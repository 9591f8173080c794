#!/usr/bin/env python
"""The bandwidth-bound kernels of the Newton step at BASELINE sizes, outside a solve, for ncu captures
and CUDA-event timings: K6 slack GEMV (C4: 250000 x 10002 = 20 GB operator), K5 triangular solves and
K3 Cholesky (m = 10001 and 20000), K7 two-sided Lanczos (n = 2000), K8 Pade geodesic update (n = 2000).

  python tools/prof_hbm_kernels.py time          # CUDA-event timings + achieved GB/s / TFLOP/s (JSON lines)
  ncu --set full --clock-control none -k regex:'GemvN|TrsvFwd|TrsvBwd|LanczosStep' -c 12 \\
      -o gpurun_out/hbm python tools/prof_hbm_kernels.py once
"""
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import conex_b200.binding as dev  # noqa: E402
import torch  # noqa: E402

L = dev.product().lib
vp = C.c_void_p
f64 = dict(dtype=torch.float64, device="cuda")


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(min(ts))


def main():
    mode = sys.argv[1] if len(sys.argv) > 1 else "time"
    # creating a program sets the release threshold of the stream-ordered pool the solves take their
    # scratch from (host/device_runtime.h); without it every call re-acquires the memory from the driver
    keep = dev.product().program()  # noqa: F841
    reps = 1 if mode == "once" else 5
    which = sys.argv[2].split(",") if len(sys.argv) > 2 else ["gemv", "chol", "lanczos", "geo"]
    s = torch.cuda.current_stream().cuda_stream
    out = []

    if "gemv" in which:
        prof_gemv(s, reps, out)
    if "chol" in which:
        prof_chol(s, reps, out, (10001,) if mode == "once" else (2000, 10001, 20000))
    if "lanczos" in which or "geo" in which:
        prof_psd(s, reps, out, which)
    for o in out:
        print(json.dumps(o))


def prof_gemv(s, reps, out):
    # K6: -S = sum y_i A_i - k C as one GEMV over the n^2 x (m + 1) operator (C4 shape)
    nn, cols = 500 * 500, 10002
    A = torch.rand(cols, nn, **f64)
    y = torch.rand(cols, **f64)
    S = torch.empty(nn, **f64)
    med, best = timed(lambda: L.cxb_gemv_n(vp(s), nn, cols, vp(A.data_ptr()), vp(y.data_ptr()), vp(S.data_ptr())), reps)
    out.append(dict(kernel="K6 cxb_gemv_n", shape=f"{nn} x {cols}", ms=med, best_ms=best,
                    algorithmic_bytes=8.0 * nn * cols, GBps=8.0 * nn * cols / (best * 1e-3) / 1e9))


def prof_chol(s, reps, out, sizes):
    # K3 + K5: Cholesky and the two triangular sweeps (L read once forward, once backward)
    for m in sizes:
        ld = m + 2 + (m % 2)
        H = torch.rand(m, ld, **f64) * 0.01
        H[:, :m] += torch.eye(m, **f64) * (0.02 * m)
        Hwork = torch.empty_like(H)
        info = torch.zeros(4, dtype=torch.int32, device="cuda")

        def factor():
            Hwork.copy_(H)
            L.cxb_potrf_lower(vp(s), m, vp(Hwork.data_ptr()), ld, None, vp(info.data_ptr()))

        def copy_only():
            Hwork.copy_(H)

        medc, bestc = timed(copy_only, reps)
        medf, bestf = timed(factor, reps)
        assert int(info.cpu()[0]) == 0
        t = bestf - bestc
        out.append(dict(kernel="K3 cxb_potrf_lower", shape=f"m = {m}", ms=t,
                        algorithmic_flops=m ** 3 / 3.0, TFLOPs=m ** 3 / 3.0 / (t * 1e-3) / 1e12))
        x = torch.rand(m, **f64)
        reps_solve = max(reps, 5 if reps > 1 else 1) * (4 if reps > 1 else 1)
        med, best = timed(lambda: L.cxb_potrs_lower(vp(s), m, vp(Hwork.data_ptr()), ld, vp(x.data_ptr()), m, 1), reps_solve)
        # launches: sentinel fill + forward sweep, sentinel fill + backward sweep
        out.append(dict(kernel="K5 cxb_potrs_lower", shape=f"m = {m}, 1 rhs", ms=med, best_ms=best,
                        algorithmic_bytes=8.0 * m * m, GBps=8.0 * m * m / (best * 1e-3) / 1e9, launches=4))
        del H, Hwork, x
        torch.cuda.empty_cache()



def prof_psd(s, reps, out, which):
    # K7: n/2 two-sided Lanczos steps, 2 matvecs of n^2 doubles each (L2-resident at n = 2000)
    n = 2000
    rng = np.random.default_rng(n)
    R = rng.standard_normal((n, n))
    W = R @ R.T / n + np.eye(n)
    Sm = rng.standard_normal((n, n))
    Sm = (Sm + Sm.T) / np.sqrt(n)
    dWS, dW, dr = dev.to_dev(W @ Sm), dev.to_dev(W), dev.to_dev(rng.standard_normal(n))
    it = n // 2
    alpha, beta, count = dev.dzeros(it + 2), dev.dzeros(it + 2), dev.izeros(2)
    work = dev.dzeros(L.cxb_lanczos_worksize(n))
    stream = torch.cuda.Stream()
    if "lanczos" not in which:
        steps = 0
    with torch.cuda.stream(stream):
        med, best = timed(lambda: L.cxb_lanczos_two_sided(vp(stream.cuda_stream), n, dev.ptr(dWS), dev.ptr(dW),
                                                          dev.ptr(dr), None, it, dev.ptr(alpha), dev.ptr(beta),
                                                          dev.ptr(count), dev.ptr(work)), reps)
    steps = int(count.cpu()[0]) + 1
    out.append(dict(kernel="K7 cxb_lanczos_two_sided (graph replay)", shape=f"n = {n}, {steps} steps", ms=med,
                    best_ms=best, us_per_step=best * 1e3 / steps, algorithmic_bytes=steps * 2 * 8.0 * n * n,
                    GBps=steps * 2 * 8.0 * n * n / (best * 1e-3) / 1e9, note="operands are L2-resident (2 x 32 MB)"))
    if "geo" not in which:
        return
    # K8: Pade geodesic update (3 GEMMs + LU + 2 triangular solves with n rhs + E W)
    Wd = dev.to_dev(W)
    WSd = dev.to_dev(0.01 * (W @ Sm))
    W0, WS0 = Wd.clone(), WSd.clone()
    gw = dev.dzeros(L.cxb_geodesic_worksize(n))
    iw = dev.izeros(2 * n + 8)
    inf = dev.izeros(4)

    def geo():
        Wd.copy_(W0)
        WSd.copy_(WS0)
        L.cxb_geodesic_update(vp(s), n, dev.ptr(Wd), dev.ptr(WSd), 0.0, 1.0, dev.ptr(gw), dev.ptr(iw), dev.ptr(inf))

    med, best = timed(geo, reps)
    out.append(dict(kernel="K8 cxb_geodesic_update (Pade + LU)", shape=f"n = {n}", ms=med, best_ms=best,
                    algorithmic_flops=10.7 * n ** 3, TFLOPs=10.7 * n ** 3 / (best * 1e-3) / 1e12))


if __name__ == "__main__":
    main()
