#!/usr/bin/env python
"""Iteration logs of BASELINE config 1 (n = 50, m = 100): oracle (BLAS and plain-loop summation) and the
device, side by side — how far the per-step trajectory is determined at all
(see tests/test_gpu_solve.py::oracle_trajectory_horizon). Then the accuracy of the device's Cholesky and
solve against an extended-precision reference on ill-conditioned matrices."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import devlib  # noqa: E402
from harness import oracle, random_dense_lmi  # noqa: E402

mats, Cm = random_dense_lmi(50, 100, 1)
ora = oracle()
dev = devlib.product()

logs = {}
for name, L, setup in (("oracle/blas", ora, lambda: ora.lib.ORACLE_ForcePlainLoops(0)),
                       ("oracle/loops", ora, lambda: ora.lib.ORACLE_ForcePlainLoops(1)),
                       ("device", dev, lambda: None)):
    setup()
    P = L.program()
    P.add_dense_lmi(mats, Cm)
    P.maximize(P.feasible_objective(), L.default_config(prepare_dual_variables=1))
    logs[name] = P.iteration_log()
ora.lib.ORACLE_ForcePlainLoops(0)
names = list(logs)
print("step " + " ".join(f"{n:>28s}" for n in names))
for i in range(max(len(v) for v in logs.values())):
    row = []
    for n in names:
        r = logs[n][i] if i < len(logs[n]) else None
        row.append(f"{r['inv_sqrt_mu']:14.6f} {r['d_inf']:6.3f} {r['by']:.6f}" if r else " " * 28)
    print(f"{i:3d}  " + " ".join(f"{x:>28s}" for x in row))


# ---- accuracy of the factorisation and the solves on an ill-conditioned Schur complement -------------
import numpy as np  # noqa: E402
import torch  # noqa: E402


def reference_cholesky(H):
    """Cholesky in 80-bit extended precision (numpy longdouble), column by column."""
    n = H.shape[0]
    Lx = np.zeros((n, n), dtype=np.longdouble)
    Hx = H.astype(np.longdouble)
    for j in range(n):
        d = Hx[j, j] - np.dot(Lx[j, :j], Lx[j, :j])
        Lx[j, j] = np.sqrt(d)
        Lx[j + 1:, j] = (Hx[j + 1:, j] - Lx[j + 1:, :j] @ Lx[j, :j]) / Lx[j, j]
    return Lx


for m, cond in ((100, 1e4), (100, 1e10), (300, 1e10), (1000, 1e8)):
    rng = np.random.default_rng(m)
    Q, _ = np.linalg.qr(rng.standard_normal((m, m)))
    ev = np.logspace(0, -np.log10(cond), m)
    H = (Q * ev) @ Q.T
    H = 0.5 * (H + H.T)
    Lx = reference_cholesky(H)
    xtrue = rng.standard_normal(m)
    b = (H.astype(np.longdouble) @ xtrue.astype(np.longdouble)).astype(np.float64)
    xref = np.linalg.solve(H, b)
    line = [f"m={m} cond={cond:.0e}: LAPACK |L-Lx|={np.abs(np.linalg.cholesky(H) - Lx).max():.2e} "
            f"x-err {np.abs(xref - xtrue).max():.2e}"]
    dH = devlib.to_dev(np.tril(H))
    info = devlib.izeros(1)
    assert dev.lib.cxb_potrf_lower(None, m, devlib.ptr(dH), m, None, devlib.ptr(info)) == 0
    Ld = np.tril(devlib.from_dev(dH))
    dx = devlib.to_dev(b)
    assert dev.lib.cxb_potrs_lower(None, m, devlib.ptr(dH), m, devlib.ptr(dx), m, 1) == 0
    xd = devlib.from_dev(dx)
    line.append(f"device: info={int(info.cpu()[0])} |L-Lx|={np.abs(Ld - Lx).max():.2e} "
                f"x-err {np.abs(xd - xtrue).max():.2e}")
    print(" | ".join(line))
