"""workloads.mpc_problem without equality blocks (eq_rows = 0): the long-horizon Cholesky workload of
tools/batch_long_horizon_bench.py. The equality blocks are drawn after the cones, so the cones do not change."""
import numpy as np

from conex_b200.workloads import mpc_problem


def test_mpc_problem_without_equality_blocks():
    cones, padded, b = mpc_problem(5, stages=29, eq_rows=0)
    with_eq, _, _ = mpc_problem(5, stages=29)
    assert b.size == 174
    assert all(entry[0] != "eq" for entry in cones + padded)
    assert len(cones) == 29 * 2 + 28
    same = [entry for entry in with_eq if entry[0] != "eq"]
    assert len(same) == len(cones)
    for x, y in zip(cones, same):
        assert x[0] == y[0] and x[3] == y[3]
        for u, v in zip(x[1:3], y[1:3]):
            assert np.array_equal(np.asarray(u), np.asarray(v))
