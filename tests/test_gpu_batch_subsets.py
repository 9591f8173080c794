"""Batched solves of programs whose cones act on subsets of the variables (dense LMIs through
CONEX_AddSparseLMIConstraint, LP and second-order cones through CONEXB200_AddSparseLinearConstraint /
CONEXB200_AddSparseSocConstraint). Every program of a batch must reproduce what the CPU oracle computes for the
zero-padded equivalent (every cone on all variables; the oracle has no LP / SOC subset entry points) and what
CONEX_Maximize computes on the device for the same subset program, with the tolerances of
test_gpu_batch_equality.py: same solved flag, iteration count within +-1, objectives within 1e-7 relative (or 10 x the
oracle's one-ulp sensitivity where larger), y within 1e-6.
"""
import ctypes as C

import numpy as np
import pytest

from harness import Batch, add_cones, dptr, mpc_problem, oracle, pad_cones, random_sym

pytestmark = pytest.mark.gpu
WARM = dict(initialization_mode=1)


@pytest.fixture(scope="module")
def libs():
    import devlib
    return oracle(), devlib.product()


def subset_problem(seed, m, spec, y0_scale=0.05):
    """A strictly feasible program of the constraints `spec`: (kind, order, variables or None = all) for cones, ("eq",
    rows, variables or None) for equality blocks. LP: A uniform, c = 1; SOC: A uniform, c = e_0; LMI: A_i = sym(U[-1,1]),
    C = I. b = sum over cones of AW/2 at W = I, plus A_eq^T lambda0; b_eq = A_eq y0[variables] at an interior y0.
    Returns (cones in the add_cones format, b)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    b = np.zeros(m)
    cones, eqs = [], []
    for kind, order, variables in spec:
        v = list(range(m)) if variables is None else list(variables)
        k = len(v)
        if kind == "eq":
            eqs.append((len(cones) + len(eqs), order, variables))
            continue
        if kind == "lp":
            A = rng.uniform(-1.0, 1.0, size=(order, k))
            entry = ("lp", A, np.ones(order))
            np.add.at(b, v, 0.5 * A.sum(axis=0))
        elif kind == "soc":
            A = rng.uniform(-1.0, 1.0, size=(order + 1, k))
            c = np.zeros(order + 1)
            c[0] = 1.0
            entry = ("soc", A, c)
            np.add.at(b, v, A[0, :])
        else:
            mats = [random_sym(rng, order) for _ in v]
            entry = ("psd", mats, np.eye(order))
            np.add.at(b, v, 0.5 * np.array([np.trace(M) for M in mats]))
        cones.append(entry if variables is None else entry + (v,))
    y0 = y0_scale * rng.uniform(-1.0, 1.0, size=m)

    def interior(y):
        for entry in cones:
            kind, A, c = entry[:3]
            yv = y if len(entry) == 3 else y[entry[3]]
            if kind == "psd":
                ok = np.linalg.eigvalsh(c - sum(yi * Ai for yi, Ai in zip(yv, A))).min() > 0.1
            elif kind == "soc":
                s = c - A @ yv
                ok = s[0] - np.linalg.norm(s[1:]) > 0.1
            else:
                ok = (c - A @ yv).min() > 0.1
            if not ok:
                return False
        return True

    while not interior(y0):
        y0 *= 0.5
    for position, rows, variables in eqs:
        v = list(range(m)) if variables is None else list(variables)
        A_eq = rng.uniform(-1.0, 1.0, size=(rows, len(v)))
        np.add.at(b, v, A_eq.T @ rng.uniform(-1.0, 1.0, size=rows))
        cones.insert(position, ("eq", A_eq, (A_eq @ y0[v], None if variables is None else v)))
    return cones, b


def make_program(L, m, cones):
    P = L.program(m)
    add_cones(P, cones)
    return P


def make_batch(D, m, probs):
    return Batch(D, [make_program(D, m, cones) for cones, _ in probs])


def oracle_reference(O, m, cones, b, cfg_kw, spread=True):
    """The oracle on the zero-padded program; with the one-ulp spread of its objectives (perturbations of b)."""
    padded = pad_cones(cones, m)
    P = make_program(O, m, padded)
    solved, y = P.maximize(b, O.default_config(**cfg_kw))
    log = P.iteration_log()
    sp = dict(by=0.0, cx=0.0)
    for j in ((-2, -1, 1, 2) if spread else ()):
        Pp = make_program(O, m, padded)
        Pp.maximize(b * (1 + j * 2.0 ** -52), O.default_config(**cfg_kw))
        lp = Pp.iteration_log()
        if len(lp) == len(log):
            for key in sp:
                sp[key] = max(sp[key], abs(lp[-1][key] - log[-1][key]))
    return solved, y, log, sp, P


def assert_parity(got, log, y_ref, solved_ref, spread=None, tag=None):
    """got = (solved, iterations, by, cx, y) of one program of the batch."""
    solved, its, by, cx, y = got
    assert solved == solved_ref, tag
    assert abs(int(its) - len(log)) <= 1, (tag, its, len(log))
    if log and int(its) == len(log):
        for name, value in (("by", by), ("cx", cx)):
            tol = max(1e-7 * max(1.0, abs(log[-1][name])), 10 * (spread or {}).get(name, 0.0))
            assert abs(value - log[-1][name]) <= tol, (tag, name, value, log[-1][name])
    assert np.abs(y - y_ref).max() <= 1e-6 * max(1.0, np.abs(y_ref).max()), tag


def batch_outcome(batch, solved, y):
    its, by, cx, _ = batch.results()
    return [(solved[p], its[p], by[p], cx[p], y[p]) for p in range(batch.count)]


def check_both_references(O, D, m, probs, cfg_kw, got):
    """Per program: the oracle on the padded program (the one-ulp spread is only computed when the plain tolerance is
    not met) and CONEX_Maximize on the device with the same subset program."""
    for p, (cones, pb) in enumerate(probs):
        so, yo, lo, _, _ = oracle_reference(O, m, cones, pb, cfg_kw, spread=False)
        try:
            assert_parity(got[p], lo, yo, so, tag=("oracle", p))
        except AssertionError:
            so, yo, lo, sp, _ = oracle_reference(O, m, cones, pb, cfg_kw)
            assert_parity(got[p], lo, yo, so, sp, tag=("oracle", p))
        Q = make_program(D, m, cones)
        sd, yd = Q.maximize(pb, D.default_config(**cfg_kw))
        assert_parity(got[p], Q.iteration_log(), yd, sd, tag=("device", p))


def solve_batch(D, m, probs, cfg_kw):
    batch = make_batch(D, m, probs)
    solved, y = batch.maximize(np.stack([pb for _, pb in probs]), D.default_config(**cfg_kw))
    return batch, solved, y


M = 6
SPECS = {
    # each cone type alone: an unsorted list, its complement, and a one-variable cone
    "lp_only": [("lp", 5, [5, 1, 3]), ("lp", 4, [0, 2, 4]), ("lp", 2, [2])],
    "soc_only": [("soc", 3, [5, 1, 3]), ("soc", 4, [0, 2, 4]), ("soc", 2, [2])],
    "psd_only": [("psd", 4, [5, 1, 3]), ("psd", 4, [0, 2, 4]), ("psd", 4, [2])],
    # mixes
    "full_first": [("psd", 4, None), ("lp", 5, [5, 1, 3]), ("soc", 3, [0, 2]), ("psd", 4, [4, 0])],
    "full_after": [("lp", 6, [1, 3]), ("soc", 3, [5, 0, 2]), ("psd", 4, None), ("lp", 4, [4])],
    "no_full": [("lp", 6, [0, 1, 2]), ("soc", 3, [3, 4, 5]), ("psd", 4, [5, 2, 0, 3]), ("lp", 3, [1, 4])],
    # equality blocks (the LDL^T path), one of them on a subset
    "no_full_eq": [("lp", 6, [0, 1, 2]), ("eq", 2, [1, 4, 5]), ("soc", 3, [3, 4, 5]), ("psd", 4, [5, 2, 0, 3]),
                   ("lp", 3, [1, 4]), ("eq", 1, None)],
    "full_first_eq": [("psd", 4, None), ("lp", 5, [5, 1, 3]), ("eq", 2, [3, 0]), ("soc", 3, [0, 2])],
}


def problems(spec, count, seed0):
    return [subset_problem(seed0 + p, M, SPECS[spec]) for p in range(count)]


@pytest.mark.parametrize("spec", ["lp_only", "soc_only", "psd_only", "full_first", "full_after", "no_full"])
def test_subset_cones_match_both_references(libs, spec):
    O, D = libs
    probs = problems(spec, 5, 100)
    batch, solved, y = solve_batch(D, M, probs, {})
    check_both_references(O, D, M, probs, {}, batch_outcome(batch, solved, y))
    assert solved.all()


@pytest.mark.parametrize("spec", ["no_full_eq", "full_first_eq"])
def test_subset_cones_with_equalities_and_dual_variables(libs, spec):
    """Equality blocks on subsets (the batched LDL^T), prepare_dual_variables = 1: results against both references,
    and the cones' dual variables against CONEX_GetDualVariable of the oracle's padded program and of the device."""
    O, D = libs
    cfg_kw = dict(prepare_dual_variables=1)
    probs = problems(spec, 4, 200)
    batch, solved, y = solve_batch(D, M, probs, cfg_kw)
    check_both_references(O, D, M, probs, cfg_kw, batch_outcome(batch, solved, y))
    assert solved.all()
    for p, (cones, pb) in enumerate(probs):
        P = make_program(O, M, pad_cones(cones, M))
        P.maximize(pb, O.default_config(**cfg_kw))
        Q = make_program(D, M, cones)
        Q.maximize(pb, D.default_config(**cfg_kw))
        for ci, entry in enumerate(cones):
            if entry[0] in ("eq", "soc"):  # equality blocks have none; the reference's SOC dual is an unset dummy
                continue
            for ref in (P, Q):
                xo = ref.dual_variable(ci)
                xd = batch.dual_variable(p, ci, xo.size).reshape(xo.shape, order="F")
                assert np.abs(xo - xd).max() <= 1e-5 * max(1.0, np.abs(xo).max()), (p, ci)
        for entry in cones:  # the equalities hold at the solution
            if entry[0] == "eq":
                A, (b_eq, v) = entry[1], entry[2]
                yv = y[p] if v is None else y[p][v]
                assert np.abs(A @ yv - b_eq).max() <= 1e-6 * max(1.0, np.abs(b_eq).max())


def test_mpc_shaped_programs(libs):
    """The generator of the benchmark (8 stages of 6 variables: per stage an LP and a second-order cone, per pair of
    stages an LMI of order 8 and a 4-row equality block; 23 cones, KKT order 76) at 64 programs; and the zero-padded
    batch of the same programs gives the same answers."""
    O, D = libs
    gen = [mpc_problem(300 + p) for p in range(64)]
    probs = [(cones, b) for cones, _, b in gen]
    m = probs[0][1].size
    assert make_program(D, m, probs[0][0]).kkt_size() == 76
    batch, solved, y = solve_batch(D, m, probs, {})
    check_both_references(O, D, m, probs, {}, batch_outcome(batch, solved, y))
    assert solved.all()
    padded, solved_p, y_p = solve_batch(D, m, [(pc, b) for _, pc, b in gen], {})
    assert (solved_p == solved).all()
    assert np.abs(y - y_p).max() <= 1e-6 * max(1.0, np.abs(y_p).max())


@pytest.mark.parametrize("spec", [
    [("lp", 5, [5, 1, 3]), ("soc", 3, [0, 2])],                  # variable 4 is in no cone: a failed Cholesky
    [("psd", 4, [5, 1, 3]), ("eq", 2, [0, 2]), ("lp", 4, [0, 2])],  # ... with equality multipliers: the LDL^T
])
def test_variable_in_no_cone(libs, spec):
    """The batch reports for every program what CONEX_Maximize reports for it."""
    O, D = libs
    probs = [subset_problem(400 + p, M, spec) for p in range(4)]
    batch, solved, y = solve_batch(D, M, probs, {})
    its = batch.results()[0]
    multipliers = any(s[0] == "eq" for s in spec)
    for p, (cones, pb) in enumerate(probs):
        Q = make_program(D, M, cones)
        sd, yd = Q.maximize(pb)
        assert solved[p] == sd, p
        assert abs(int(its[p]) - len(Q.iteration_log())) <= 1, p
        if not multipliers:
            assert sd == 0
            so, _ = make_program(O, M, pad_cones(cones, M)).maximize(pb)
            assert so == 0


def create_batch(D, programs):
    L = D.lib
    L.CONEXB200_CreateBatch.restype = C.c_void_p
    L.CONEXB200_CreateBatch.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    handles = (C.c_void_p * len(programs))(*[q.h for q in programs])
    return L.CONEXB200_CreateBatch(handles, len(programs))


@pytest.mark.parametrize("other", [
    [("lp", 5, [1, 3, 5]), ("soc", 3, [0, 2, 4])],     # the same variables in another order
    [("lp", 5, [5, 1, 2]), ("soc", 3, [0, 3, 4])],     # other variables
    [("lp", 5, None), ("soc", 3, [0, 2, 4])],          # all variables
    [("lp", 5, [5, 1, 3, 0]), ("soc", 3, [0, 2, 4])],  # more variables
])
def test_batch_rejects_different_variable_lists(libs, other):
    _, D = libs
    base = [("lp", 5, [5, 1, 3]), ("soc", 3, [0, 2, 4])]
    ca, _ = subset_problem(1, M, base)
    cb, _ = subset_problem(2, M, other)
    assert not create_batch(D, [make_program(D, M, ca), make_program(D, M, cb)])
    cc, _ = subset_problem(3, M, base)
    h = create_batch(D, [make_program(D, M, ca), make_program(D, M, cc)])
    assert h
    D.lib.CONEXB200_DeleteBatch.argtypes = [C.c_void_p]
    D.lib.CONEXB200_DeleteBatch(h)


# ---- in-place updates of subset cones ---------------------------------------------------------------------------

def data_matrix(entry):
    """[A | c] of a cone on m_k variables (LMI: vec(A_j), vec(C)): m_k + 1 columns."""
    kind, A, c = entry[:3]
    if kind == "psd":
        return np.stack([Mj.ravel(order="F") for Mj in A] + [c.ravel(order="F")], axis=1)
    return np.column_stack([A, c])


def from_data_matrix(entry, X):
    kind, A, c, v = entry
    if kind == "psd":
        n = c.shape[0]
        mats = [X[:, j].reshape((n, n), order="F") for j in range(X.shape[1] - 1)]
        return kind, mats, X[:, -1].reshape((n, n), order="F"), v
    return kind, X[:, :-1].copy(), X[:, -1].copy(), v


def updated(probs, constraint, first, count, seed, scale):
    rng = np.random.Generator(np.random.PCG64(seed))
    out, blocks = [], []
    for cones, pb in probs:
        entry = cones[constraint]
        X = data_matrix(entry)
        noise = rng.uniform(-1.0, 1.0, size=(X.shape[0], count))
        if entry[0] == "psd":
            n = entry[2].shape[0]
            noise = np.stack([(0.5 * (N + N.T)).ravel(order="F")
                              for N in (noise[:, j].reshape((n, n), order="F") for j in range(count))], axis=1)
        X[:, first:first + count] += scale * noise
        blocks.append(X[:, first:first + count])
        new = list(cones)
        new[constraint] = from_data_matrix(entry, X)
        out.append((new, pb))
    return out, np.stack(blocks)


# spec no_full: LP 6 x [0, 1, 2], SOC 3 on [3, 4, 5], LMI 4 on [5, 2, 0, 3], LP 3 x [1, 4]
@pytest.mark.parametrize("constraint,first,count", [(0, 0, 4), (1, 2, 2), (2, 1, 4), (3, 2, 1)])
def test_update_of_a_subset_cone(libs, constraint, first, count):
    """The shape reports m_k + 1 columns; an update followed by a cold solve equals a freshly built batch of the new
    data bit for bit; an update followed by a warm solve matches a single-program warm solve on the old program's
    memory."""
    _, D = libs
    probs = problems("no_full", 4, 500)
    rows_cols = [(6, 4), (4, 4), (16, 5), (3, 3)][constraint]
    new, blocks = updated(probs, constraint, first, count, 501, 0.01)
    b = np.stack([pb for _, pb in probs])
    cfg = D.default_config(prepare_dual_variables=1)
    batch = make_batch(D, M, probs)
    rows, columns = C.c_int(), C.c_int()
    assert D.lib.CONEXB200_BatchConstraintDataShape(batch.h, constraint, C.byref(rows), C.byref(columns)) == 0
    assert (rows.value, columns.value) == rows_cols
    f = D.lib.CONEXB200_BatchUpdateConstraintData
    assert f(batch.h, constraint, columns.value - 1, 2, dptr(np.zeros(4 * rows.value * 2))) == -1
    batch.maximize(b, cfg)
    batch.update(constraint, first, blocks)
    solved, y = batch.maximize(b, cfg)
    fresh = make_batch(D, M, new)
    solved_f, y_f = fresh.maximize(b, cfg)
    assert (solved == solved_f).all()
    assert np.array_equal(y, y_f, equal_nan=True)
    for got, want in zip(batch.results()[:3], fresh.results()[:3]):
        assert np.array_equal(got, want, equal_nan=True)

    warm = make_batch(D, M, probs)
    warm.maximize(b)
    warm.update(constraint, first, blocks)
    solved_w, y_w = warm.maximize(b, D.default_config(**WARM))
    got = batch_outcome(warm, solved_w, y_w)
    for p, ((cones, pb), (new_cones, _)) in enumerate(zip(probs, new)):
        Q = make_program(D, M, cones)
        Q.maximize(pb)
        Q2 = D.program_on_memory_of(Q, M)
        add_cones(Q2, new_cones)
        s2, y2 = Q2.maximize(pb, D.default_config(**WARM))
        assert_parity(got[p], Q2.iteration_log(), y2, s2, tag=p)
        del Q2  # before Q: it lives on Q's memory


# ---- the entry points on single programs ------------------------------------------------------------------------

def test_sparse_linear_and_soc_entry_points(libs):
    """CONEXB200_AddSparseLinearConstraint / CONEXB200_AddSparseSocConstraint through CONEX_Maximize against the
    oracle's padded program; bad variable lists return -1 and add nothing."""
    O, D = libs
    for seed, spec in enumerate([SPECS["lp_only"], SPECS["soc_only"], SPECS["no_full"]]):
        cones, b = subset_problem(600 + seed, M, spec)
        Q = make_program(D, M, cones)
        sd, yd = Q.maximize(b)
        so, yo, lo, sp, _ = oracle_reference(O, M, cones, b, {})
        assert_parity((sd, len(Q.iteration_log()), Q.iteration_log()[-1]["by"], Q.iteration_log()[-1]["cx"], yd),
                      lo, yo, so, sp, tag=seed)
        assert sd == 1
    L = D.lib
    L.CONEXB200_NumberOfConstraints.argtypes = [C.c_void_p]
    P = D.program(M)
    A = np.asfortranarray(np.ones((3, 2)))
    c = np.ones(3)
    for bad in ([1, 1], [0, 6], [-1, 2]):
        v = (C.c_long * 2)(*bad)
        assert L.CONEXB200_AddSparseLinearConstraint(P.h, dptr(A), 3, 2, dptr(c), v) == -1, bad
        assert L.CONEXB200_AddSparseSocConstraint(P.h, 2, 2, dptr(A), dptr(c), v) == -1, bad
        assert L.CONEXB200_NumberOfConstraints(P.h) == 0
    v = (C.c_long * 2)(4, 1)
    assert L.CONEXB200_AddSparseLinearConstraint(P.h, dptr(A), 3, 2, dptr(c), v) == 0
    assert L.CONEXB200_AddSparseSocConstraint(P.h, 2, 2, dptr(A), dptr(c), v) == 1
    assert L.CONEXB200_NumberOfConstraints(P.h) == 2
