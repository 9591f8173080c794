"""The MPC-shaped generator (conex_b200.workloads.mpc_problem) and pad_cones, on the CPU: shape, strict feasibility
by construction, and the padded program acting on y exactly like the subset program."""
import numpy as np

from harness import mpc_problem, pad_cones


def test_mpc_problem_shape():
    cones, padded, b = mpc_problem(1)
    m = b.size
    assert m == 48
    kinds = [entry[0] for entry in cones]
    assert kinds.count("lp") == 8 and kinds.count("soc") == 8 and kinds.count("psd") == 7 and kinds.count("eq") == 7
    assert sum(entry[1].shape[0] for entry in cones if entry[0] == "eq") == 28  # KKT order 48 + 28 = 76
    for entry in cones:
        kind, A, c = entry[:3]
        v = entry[3] if kind != "eq" else c[1]
        assert len(set(v)) == len(v) and min(v) >= 0 and max(v) < m
        assert len(v) == (12 if kind in ("psd", "eq") else 6)
        if kind == "psd":
            assert len(A) == 12 and c.shape == (8, 8)
        elif kind == "soc":
            assert A.shape == (7, 6)
        elif kind == "lp":
            assert A.shape == (12, 6)
    assert [e[0] for e in padded] == kinds
    again = mpc_problem(1)
    assert np.array_equal(again[2], b)


def test_mpc_problem_is_strictly_feasible_and_padding_preserves_it():
    """b = sum of AW/2 at W = I plus A_eq^T lambda for some lambda (checked as: b minus the cone part lies in the range
    of the stacked A_eq^T), and the padded cones act on y like the subset cones."""
    cones, padded, b = mpc_problem(7)
    m = b.size
    rng = np.random.default_rng(0)
    y = rng.uniform(-1.0, 1.0, size=m)
    cone_part = np.zeros(m)
    eq_cols = []
    for entry, pe in zip(cones, padded):
        kind, A, c = entry[:3]
        if kind == "eq":
            col = np.zeros((m, A.shape[0]))
            col[c[1], :] = A.T
            eq_cols.append(col)
            assert pe[0] == "eq"
            continue
        v = entry[3]
        assert len(pe) == 3
        if kind == "psd":
            assert np.allclose(sum(yi * Ai for yi, Ai in zip(y[v], A)), sum(yi * Ai for yi, Ai in zip(y, pe[1])))
            np.add.at(cone_part, v, 0.5 * np.array([np.trace(Mj) for Mj in A]))
        else:
            assert np.allclose(pe[1] @ y, A @ y[v], rtol=0, atol=1e-13)
            np.add.at(cone_part, v, 0.5 * A.sum(axis=0) if kind == "lp" else A[0, :])
    E = np.hstack(eq_cols)
    lam, *_ = np.linalg.lstsq(E, b - cone_part, rcond=None)
    assert np.abs(E @ lam - (b - cone_part)).max() < 1e-10
    # the equality blocks are consistent with each other
    A_all = np.vstack([_eq_rows(entry, m) for entry in cones if entry[0] == "eq"])
    b_all = np.concatenate([entry[2][0] for entry in cones if entry[0] == "eq"])
    y0, *_ = np.linalg.lstsq(A_all, b_all, rcond=None)
    assert np.abs(A_all @ y0 - b_all).max() < 1e-10


def _eq_rows(entry, m):
    A, (_, v) = entry[1], entry[2]
    out = np.zeros((A.shape[0], m))
    out[:, v] = A
    return out


def test_pad_cones_keeps_full_cones_and_equalities():
    A = np.ones((2, 3))
    cones = [("lp", A, np.ones(2)), ("eq", A, (np.ones(2), [0, 1, 2])), ("soc", A, np.ones(2), [2, 0, 1])]
    out = pad_cones(cones, 3)
    assert out[0] == cones[0] and out[1] == cones[1]
    assert np.array_equal(out[2][1], A)  # the columns of the variables 2, 0, 1, all ones
