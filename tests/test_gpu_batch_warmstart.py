"""Warm starts and in-place data updates of batched solves (CONEXB200_BatchMaximize with initialization_mode = 1,
CONEXB200_BatchUpdateConstraintData). A warm-started program of a batch must follow the sequence it follows alone
through CONEX_Maximize on the same memory — and match the CPU oracle warm-starting the same handle — with the
tolerances of test_gpu_batch.py: same solved flag, iteration count within +-1, objectives within 1e-7 relative (or
10 x the oracle's one-ulp sensitivity where larger), y within 1e-6. An update followed by a cold solve must give what
a batch built from the new data gives, bit for bit.
"""
import ctypes as C

import numpy as np
import pytest

from harness import Batch, add_cones, dptr, oracle, small_multicone_equality_problem, small_multicone_problem

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def libs():
    import devlib
    return oracle(), devlib.product()


SHAPES = {
    "tiny": dict(m=5, psd_blocks=1, psd_order=4, soc_cones=1, soc_order=3, lp_rows=6),
    "mixed": dict(m=8, psd_blocks=2, psd_order=6, soc_cones=2, soc_order=4, lp_rows=8),
    "c3": dict(m=40, psd_blocks=3, psd_order=20, soc_cones=2, soc_order=10, lp_rows=40),
}
# case -> (shape, equality blocks or None); constraint order: LMI blocks, second-order cones, the LP block, then the
# equality block
CASES = {"tiny": ("tiny", None), "mixed": ("mixed", None), "tiny_eq": ("tiny", ((2, None, None),)),
         "c3": ("c3", None)}
WARM = dict(initialization_mode=1)


def problems(case, count, seed0):
    shape, eqs = CASES[case]
    kw = SHAPES[shape]
    if eqs is None:
        return kw["m"], [small_multicone_problem(seed0 + p, **kw) for p in range(count)]
    return kw["m"], [small_multicone_equality_problem(seed0 + p, equalities=eqs, **kw) for p in range(count)]


def make_program(L, m, cones):
    P = L.program(m)
    add_cones(P, cones)
    return P


def make_batch(D, m, probs):
    return Batch(D, [make_program(D, m, cones) for cones, _ in probs])


def perturbed_b(probs, seed, scale=0.05):
    rng = np.random.Generator(np.random.PCG64(seed))
    b = np.stack([pb for _, pb in probs])
    return b * (1 + scale * rng.uniform(-1.0, 1.0, size=b.shape))


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


def oracle_warm(O, m, cones, b1, b2, cfg_kw):
    """The oracle solving b1 from a cold start, then b2 warm-started on the same handle; with the one-ulp spread of
    the second solve's objectives (perturbations of b2)."""
    def run(b2p):
        P = make_program(O, m, cones)
        P.maximize(b1, O.default_config(**cfg_kw))
        s, y = P.maximize(b2p, O.default_config(**cfg_kw, **WARM))
        return s, y, P.iteration_log()
    so, yo, lo = run(b2)
    spread = dict(by=0.0, cx=0.0)
    for j in (-2, -1, 1, 2):
        _, _, lp = run(b2 * (1 + j * 2.0 ** -52))
        if len(lp) == len(lo):
            for key in spread:
                spread[key] = max(spread[key], abs(lp[-1][key] - lo[-1][key]))
    return so, yo, lo, spread


def device_warm(D, m, cones, b1, b2, cfg_kw, warm_kw=None):
    """CONEX_Maximize on the device: b1 cold, then b2 warm-started on the same program."""
    Q = make_program(D, m, cones)
    Q.maximize(b1, D.default_config(**cfg_kw))
    s, y = Q.maximize(b2, D.default_config(**cfg_kw, **WARM, **(warm_kw or {})))
    return s, y, Q.iteration_log()


def batch_outcome(batch, solved, y):
    its, by, cx, _ = batch.results()
    return [(solved[p], its[p], by[p], cx[p], y[p]) for p in range(batch.count)]


# ---- warm starts ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case,count", [("tiny", 6), ("mixed", 4), ("tiny_eq", 5), ("c3", 4)])
def test_split_solve_equals_whole_solve(libs, case, count):
    """test_warmstart.cc:14-45 for a batch: one 10-iteration solve == one 1-iteration cold solve followed by nine
    1-iteration warm solves, every program within 1e-12. (No abort threshold in the split run: the whole solve
    never restarts, a 1-iteration warm solve would test its first step against it.)"""
    _, D = libs
    m, probs = problems(case, count, 100)
    b = np.stack([pb for _, pb in probs])
    kw = dict(inv_sqrt_mu_max=1e7, final_centering_steps=0)
    whole = make_batch(D, m, probs)
    _, y = whole.maximize(b, D.default_config(max_iterations=10, **kw))
    assert (whole.results()[0] == 10).all()
    split = make_batch(D, m, probs)
    for i in range(10):
        _, ys = split.maximize(b, D.default_config(max_iterations=1, initialization_mode=0 if i == 0 else 1,
                                                   warmstart_abort_threshold=1e300, **kw))
    assert np.abs(y - ys).max(axis=1).max() < 1e-12


@pytest.mark.parametrize("dual", [0, 1])
@pytest.mark.parametrize("case,count,scale", [("tiny", 6, 0.05), ("mixed", 4, 0.05), ("tiny_eq", 5, 0.05),
                                              ("c3", 3, 0.01)])
def test_warm_resolve_with_new_b(libs, case, count, scale, dual):
    """After a converged cold solve, a warm solve with a new b: per program against the oracle warm-starting the same
    handle with the same b sequence and against CONEX_Maximize on the device. With prepare_dual_variables = 1 the
    first solve's dual recovery moves the iterate the second one starts from, in all three. (C3 with b changed by 1 %:
    at 5 % the reference's own warm start needs up to 47 iterations on these programs — from a converged iterate whose
    first step stays below the abort threshold it crawls — and the comparison would sit at the iteration limit.)"""
    O, D = libs
    m, probs = problems(case, count, 200)
    b1 = np.stack([pb for _, pb in probs])
    b2 = perturbed_b(probs, 201, scale)
    cfg_kw = dict(prepare_dual_variables=dual)
    batch = make_batch(D, m, probs)
    batch.maximize(b1, D.default_config(**cfg_kw))
    solved, y = batch.maximize(b2, D.default_config(**cfg_kw, **WARM))
    got = batch_outcome(batch, solved, y)
    for p, (cones, _) in enumerate(probs):
        so, yo, lo, spread = oracle_warm(O, m, cones, b1[p], b2[p], cfg_kw)
        assert_parity(got[p], lo, yo, so, spread, ("oracle", p))
        sd, yd, ld = device_warm(D, m, cones, b1[p], b2[p], cfg_kw)
        assert_parity(got[p], ld, yd, sd, spread, ("device", p))


@pytest.mark.parametrize("case,count", [("tiny", 4), ("mixed", 4), ("tiny_eq", 4)])
def test_warm_start_from_converged_iterate(libs, case, count):
    """test_warmstart.cc:47-79: two warm steps from a converged iterate return the same y (1e-9, or twice the
    distance the oracle's own re-solve moves it where that is larger: the distance is the convergence tolerance of
    the first solve)."""
    O, D = libs
    m, probs = problems(case, count, 300)
    b = np.stack([pb for _, pb in probs])
    kw = dict(final_centering_steps=3, final_centering_tolerance=.01)
    batch = make_batch(D, m, probs)
    solved, y = batch.maximize(b, D.default_config(**kw))
    assert solved.all()
    _, y2 = batch.maximize(b, D.default_config(max_iterations=2, **kw, **WARM))
    for p, (cones, pb) in enumerate(probs):
        P = make_program(O, m, cones)
        _, yo = P.maximize(pb, O.default_config(**kw))
        _, yo2 = P.maximize(pb, O.default_config(max_iterations=2, **kw, **WARM))
        bound = max(1e-9 * max(1.0, np.abs(y[p]).max()), 2 * np.abs(yo - yo2).max())
        assert np.abs(y[p] - y2[p]).max() <= bound, (p, np.abs(y[p] - y2[p]).max(), bound)


def test_abort_threshold_zero_restarts_every_program(libs):
    """warmstart_abort_threshold = 0: every program's first step is too large, every program restarts from the
    identity (and keeps its scalings); each must match its own CONEX_Maximize run."""
    _, D = libs
    m, probs = problems("mixed", 6, 400)
    b1 = np.stack([pb for _, pb in probs])
    b2 = perturbed_b(probs, 401)
    batch = make_batch(D, m, probs)
    batch.maximize(b1)
    solved, y = batch.maximize(b2, D.default_config(warmstart_abort_threshold=0.0, **WARM))
    got = batch_outcome(batch, solved, y)
    for p, (cones, _) in enumerate(probs):
        sd, yd, ld = device_warm(D, m, cones, b1[p], b2[p], {}, dict(warmstart_abort_threshold=0.0))
        assert_parity(got[p], ld, yd, sd, tag=p)


@pytest.mark.parametrize("case,count", [("mixed", 12), ("tiny_eq", 12)])
def test_abort_threshold_that_splits_the_batch(libs, case, count):
    """A threshold between the first-step sizes of the programs: some restart, the others continue, in one batch."""
    _, D = libs
    m, probs = problems(case, count, 500)
    b1 = np.stack([pb for _, pb in probs])
    rng = np.random.Generator(np.random.PCG64(501))
    b2 = b1 * (1 + rng.uniform(0.01, 0.3, size=(count, 1)) * rng.uniform(-1.0, 1.0, size=b1.shape))
    d_inf = np.array([device_warm(D, m, cones, b1[p], b2[p], {}, dict(warmstart_abort_threshold=1e300))[2][0]["d_inf"]
                      for p, (cones, _) in enumerate(probs)])
    s = np.sort(d_inf)
    lo, hi = count // 4, 3 * count // 4  # gaps around the median
    g = lo + int(np.argmax(s[lo + 1:hi + 1] - s[lo:hi]))
    threshold = 0.5 * (s[g] + s[g + 1])
    assert (d_inf >= threshold).any() and (d_inf < threshold).any()
    batch = make_batch(D, m, probs)
    batch.maximize(b1)
    solved, y = batch.maximize(b2, D.default_config(warmstart_abort_threshold=threshold, **WARM))
    got = batch_outcome(batch, solved, y)
    for p, (cones, _) in enumerate(probs):
        sd, yd, ld = device_warm(D, m, cones, b1[p], b2[p], {}, dict(warmstart_abort_threshold=threshold))
        assert_parity(got[p], ld, yd, sd, tag=(p, d_inf[p], threshold))


# ---- in-place updates -------------------------------------------------------------------------------------------

def data_matrix(entry):
    """The columns CONEXB200_BatchUpdateConstraintData addresses: [A | c] (LMI: vec(A_j), vec(C)), [A | b]."""
    kind, A, c = entry
    if kind == "psd":
        return np.stack([M.ravel(order="F") for M in A] + [c.ravel(order="F")], axis=1)
    if kind == "eq":
        return np.column_stack([A, c[0]])
    return np.column_stack([A, c])


def from_data_matrix(entry, X):
    kind, A, c = entry
    if kind == "psd":
        n = c.shape[0]
        return kind, [X[:, j].reshape((n, n), order="F") for j in range(X.shape[1] - 1)], X[:, -1].reshape(
            (n, n), order="F")
    if kind == "eq":
        return kind, X[:, :-1].copy(), (X[:, -1].copy(), c[1])
    return kind, X[:, :-1].copy(), X[:, -1].copy()


def updated(probs, constraint, first, count, seed, scale, symmetric=True):
    """New data for columns [first, first + count) of `constraint` of every program: (new problems, blocks of shape
    (programs, rows, count)). LMI columns get symmetric perturbations unless symmetric=False."""
    rng = np.random.Generator(np.random.PCG64(seed))
    out, blocks = [], []
    for cones, pb in probs:
        entry = cones[constraint]
        X = data_matrix(entry)
        noise = rng.uniform(-1.0, 1.0, size=(X.shape[0], count))
        if entry[0] == "psd" and symmetric:
            n = entry[2].shape[0]
            noise = np.stack([(0.5 * (N + N.T)).ravel(order="F")
                              for N in (noise[:, j].reshape((n, n), order="F") for j in range(count))], axis=1)
        X[:, first:first + count] += scale * noise
        blocks.append(X[:, first:first + count])
        new = list(cones)
        new[constraint] = from_data_matrix(entry, X)
        out.append((new, pb))
    return out, np.stack(blocks)


def dual_variables(batch, probs):
    out = []
    for p, (cones, _) in enumerate(probs):
        for ci, (kind, A, c) in enumerate(cones):
            if kind != "eq":
                out.append(batch.dual_variable(p, ci, np.asarray(c).size))
    return np.concatenate(out)


@pytest.mark.parametrize("case,constraint,first,count,symmetric", [
    ("tiny", 2, 0, 6, True),        # LP: all of A and c
    ("tiny", 1, 1, 3, True),        # second-order cone: a range in the middle of A
    ("mixed", 0, 2, 4, True),       # LMI matrices A_2 .. A_5
    ("mixed", 1, 8, 1, True),       # LMI affine term C
    ("mixed", 0, 3, 2, False),      # LMI matrices that are not symmetric: the packed copy is dropped
    ("tiny_eq", 3, 0, 6, True),     # equality block: A and b
    ("tiny_eq", 3, 5, 1, True),     # equality block: b
    ("c3", 2, 10, 31, True),        # C3: LMI matrices A_10 .. A_39 and C
])
def test_update_then_cold_solve_equals_fresh_batch(libs, case, constraint, first, count, symmetric):
    _, D = libs
    m, probs = problems(case, 5, 600)
    new, blocks = updated(probs, constraint, first, count, 601, 0.05, symmetric)
    b = np.stack([pb for _, pb in probs])
    cfg = D.default_config(prepare_dual_variables=1)
    batch = make_batch(D, m, probs)
    batch.maximize(b, cfg)
    batch.update(constraint, first, blocks)
    solved, y = batch.maximize(b, cfg)
    fresh = make_batch(D, m, new)
    solved_f, y_f = fresh.maximize(b, cfg)
    assert (solved == solved_f).all()
    assert np.array_equal(y, y_f, equal_nan=True)
    for got, want in zip(batch.results()[:3], fresh.results()[:3]):
        assert np.array_equal(got, want, equal_nan=True)
    assert np.array_equal(dual_variables(batch, probs), dual_variables(fresh, new), equal_nan=True)


@pytest.mark.parametrize("case,constraint,first,count", [
    ("tiny", 2, 0, 6),        # LP: A and c
    ("mixed", 0, 8, 1),       # LMI affine term
    ("mixed", 3, 0, 9),       # a second-order cone: A and c
    ("tiny_eq", 3, 0, 6),     # equality block: A and b
])
def test_update_then_warm_solve(libs, case, constraint, first, count):
    """Per program against a program on the memory of the old one (the reference's `Program prog2(m, &prog.memory_)`)
    built with the new data and warm-started on the device; and the warm start reaches the optimum of the updated
    program (the oracle's cold solve, 1e-6)."""
    O, D = libs
    m, probs = problems(case, 4, 700)
    new, blocks = updated(probs, constraint, first, count, 701, 0.01)
    b = np.stack([pb for _, pb in probs])
    batch = make_batch(D, m, probs)
    batch.maximize(b)
    batch.update(constraint, first, blocks)
    solved, y = batch.maximize(b, D.default_config(**WARM))
    got = batch_outcome(batch, solved, y)
    for p, ((cones, pb), (new_cones, _)) in enumerate(zip(probs, new)):
        Q = make_program(D, m, cones)
        Q.maximize(pb)
        Q2 = D.program_on_memory_of(Q, m)
        add_cones(Q2, new_cones)
        s2, y2 = Q2.maximize(pb, D.default_config(**WARM))
        assert_parity(got[p], Q2.iteration_log(), y2, s2, tag=p)
        del Q2  # before Q: it lives on Q's memory
        so, yo = make_program(O, m, new_cones).maximize(pb)
        assert so == solved[p] == 1, p
        assert np.abs(y[p] - yo).max() <= 1e-6 * max(1.0, np.abs(yo).max()), p


@pytest.mark.parametrize("failing", [(0, 2), (0, 1, 2, 3)])
def test_warm_start_restarts_after_a_failed_factorisation(libs, failing):
    """A warm start whose first Cholesky fails resets that program to the identity and skips the rest of iteration 0
    (then fails again here: the programs in `failing` get variable 3 removed from every cone, so every KKT matrix has
    a zero row); the other programs of the batch carry on. Per program against a program on the memory of the old one,
    built with the new data and warm-started through CONEX_Maximize. With every program failing, both lock steps are
    still timed."""
    _, D = libs
    m, probs = problems("mixed", 4, 1200)
    b = np.stack([pb for _, pb in probs])
    new = [(list(cones), pb) for cones, pb in probs]
    batch = make_batch(D, m, probs)
    batch.maximize(b)
    for k in range(len(probs[0][0])):  # constraints: LMI, LMI, SOC, SOC, LP
        blocks = []
        for p, (cones, _) in enumerate(new):
            X = data_matrix(cones[k])
            if p in failing:
                X[:, 3] = 0.0
                cones[k] = from_data_matrix(cones[k], X)
            blocks.append(X[:, 3:4])
        batch.update(k, 3, np.stack(blocks))
    solved, y = batch.maximize(b, D.default_config(**WARM))
    got = batch_outcome(batch, solved, y)
    for p, ((cones, pb), (new_cones, _)) in enumerate(zip(probs, new)):
        Q = make_program(D, m, cones)
        Q.maximize(pb)
        Q2 = D.program_on_memory_of(Q, m)
        add_cones(Q2, new_cones)
        s2, y2 = Q2.maximize(pb, D.default_config(**WARM))
        assert_parity(got[p], Q2.iteration_log(), y2, s2, tag=p)
        del Q2
        assert (solved[p] == 0) == (p in failing), p
    if len(failing) == len(probs):
        assert (batch.results()[0] == 0).all()
        assert len(batch.step_milliseconds()) == 2  # the restart step and the step whose factorisations fail


# ---- refusals ---------------------------------------------------------------------------------------------------

def test_warm_solve_before_any_solve_is_refused(libs):
    _, D = libs
    m, probs = problems("tiny", 3, 800)
    b = np.stack([pb for _, pb in probs])
    batch = make_batch(D, m, probs)
    with pytest.raises(AssertionError, match="BatchMaximize failed"):
        batch.maximize(b, D.default_config(**WARM))
    solved, _ = batch.maximize(b)
    assert solved.all()


def test_bad_updates_are_refused_and_change_nothing(libs):
    _, D = libs
    m, probs = problems("tiny_eq", 3, 900)  # constraints: LMI 16 x 6, SOC 4 x 6, LP 6 x 6, equality 2 x 6
    b = np.stack([pb for _, pb in probs])
    batch, reference = make_batch(D, m, probs), make_batch(D, m, probs)
    f = D.lib.CONEXB200_BatchUpdateConstraintData
    data = np.zeros(3 * 16 * 7)
    for constraint, first, count in [(-1, 0, 1), (4, 0, 1), (0, -1, 2), (0, 0, 0), (0, 6, 1), (0, 3, 4), (3, 5, 2),
                                     (3, 0, 7)]:
        assert f(batch.h, constraint, first, count, dptr(data)) == -1, (constraint, first, count)
    assert f(batch.h, 0, 0, 1, None) == -1
    shape = D.lib.CONEXB200_BatchConstraintDataShape
    rows, columns = C.c_int(), C.c_int()
    for constraint, want in enumerate([(16, 6), (4, 6), (6, 6), (2, 6)]):
        assert shape(batch.h, constraint, C.byref(rows), C.byref(columns)) == 0
        assert (rows.value, columns.value) == want, constraint
    assert shape(batch.h, 4, C.byref(rows), C.byref(columns)) == -1
    with pytest.raises(AssertionError):  # the binding checks the rows before the call
        batch.update(2, 0, np.zeros((3, 5, 1)))
    solved, y = batch.maximize(b)
    solved_r, y_r = reference.maximize(b)
    assert (solved == solved_r).all() and np.array_equal(y, y_r)
    for got, want in zip(batch.results(), reference.results()):
        assert np.array_equal(got, want)


def test_existing_refusals_apply_to_warm_solves(libs):
    _, D = libs
    m, probs = problems("tiny_eq", 2, 1000)
    b = np.stack([pb for _, pb in probs])
    batch = make_batch(D, m, probs)
    batch.maximize(b)
    for kw in (dict(iterative_refinement_iterations=1), dict(kkt_solver=2)):
        with pytest.raises(AssertionError, match="BatchMaximize failed"):
            batch.maximize(b, D.default_config(**kw, **WARM))
    # a line search on programs of LP cones and equality constraints only
    rng = np.random.Generator(np.random.PCG64(1001))
    programs, bs = [], []
    for _ in range(2):
        A = rng.uniform(-1.0, 1.0, size=(8, 4))
        center = A @ (0.1 * rng.uniform(-1.0, 1.0, size=4))
        lb, ub = center - 1.0, center + 1.0
        lb[6:] = ub[6:] = center[6:]
        P = D.program(4)
        P.add_linear_inequalities(A, lb, ub)
        programs.append(P)
        bs.append(rng.uniform(-1.0, 1.0, size=4))
    lp = Batch(D, programs)
    lp.maximize(np.stack(bs))
    with pytest.raises(AssertionError, match="BatchMaximize failed"):
        lp.maximize(np.stack(bs), D.default_config(enable_line_search=1, **WARM))
    solved, _ = batch.maximize(b, D.default_config(**WARM))  # the batch stays usable
    assert solved.all()


def test_public_interface_warm_start_and_update(libs):
    """conex_b200.ConexBatch: UpdateConstraintData and initialization_mode = 1 reach the optimum of a cold solve of the
    updated programs (the public class builds LMI and LP constraints)."""
    import conex_b200
    kw = dict(m=5, psd_blocks=1, psd_order=4, soc_cones=0, soc_order=1, lp_rows=6)
    probs = [small_multicone_problem(1100 + p, **kw) for p in range(3)]
    new, blocks = updated(probs, 1, 5, 1, 1101, 0.01)  # the LP's affine term c

    def program(cones):
        P = conex_b200.Conex(kw["m"])
        (_, mats, Cm), (_, A, c) = cones
        P.AddDenseLinearMatrixInequality(np.stack(mats, axis=2), Cm)
        P.AddLinearInequality(A, c)
        return P

    b = np.stack([pb for _, pb in probs])
    batch = conex_b200.ConexBatch([program(c) for c, _ in probs])
    batch.Maximize(b)
    batch.UpdateConstraintData(1, 5, blocks)
    config = conex_b200.programs_default_configuration()
    config.initialization_mode = 1
    warm = batch.Maximize(b, config)
    cold = conex_b200.ConexBatch([program(c) for c, _ in new]).Maximize(b)
    for w, c in zip(warm, cold):
        assert w.status == c.status == 1
        assert np.abs(w.y - c.y).max() <= 1e-6 * max(1.0, np.abs(c.y).max())
    with pytest.raises(NameError):
        batch.UpdateConstraintData(2, 0, blocks)
    with pytest.raises(NameError):  # rows of the LP block: 6, not 5
        batch.UpdateConstraintData(1, 5, blocks[:, :5])
