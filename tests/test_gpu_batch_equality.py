"""Batched solves of programs with equality constraints (CONEXB200_CreateBatch / BatchMaximize with
EqualityConstraints blocks): the KKT systems carry the multipliers and are factored by the batched regularised
LDL^T (cxb_small_ldlt). Every program must reproduce what the CPU oracle — and CONEX_Maximize on the device, whose
dense LDL^T path handles the same programs one at a time — computes for it alone, with the tolerances of
test_gpu_batch.py: same solved flag, iteration count within +-1, objectives within 1e-7 relative (or 10 x the
oracle's one-ulp sensitivity where larger), y within 1e-6.
"""
import ctypes as C

import numpy as np
import pytest

from harness import Batch, add_cones, dptr, oracle, small_multicone_equality_problem

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
# (shape, equality blocks: (rows, variables or None = all, position in the constraint list or None = last))
CASES = {
    "tiny_2rows": ("tiny", ((2, None, None),)),
    "mixed_two_blocks": ("mixed", ((3, None, 0), (2, [6, 1, 4], None))),
    "c3_8rows": ("c3", ((8, None, None),)),
}


def make_program(L, m, cones):
    P = L.program(m)
    add_cones(P, cones)
    return P


def oracle_reference(O, m, cones, b, cfg_kw):
    P = make_program(O, m, cones)
    solved, y = P.maximize(b, O.default_config(**cfg_kw))
    log = P.iteration_log()
    spread = dict(by=0.0, cx=0.0)
    for j in (-2, -1, 1, 2):
        Pp = make_program(O, m, cones)
        Pp.maximize(b * (1 + j * 2.0 ** -52), O.default_config(**cfg_kw))
        lp = Pp.iteration_log()
        if len(lp) == len(log):
            for key in spread:
                spread[key] = max(spread[key], abs(lp[-1][key] - log[-1][key]))
    return solved, y, log, spread, P


def check_against_oracle(O, m, problems, solved, y, its, by, cx, cfg_kw):
    for p, (cones, pb) in enumerate(problems):
        so, yo, lo, spread, _ = oracle_reference(O, m, cones, pb, cfg_kw)
        assert solved[p] == so, p
        assert abs(int(its[p]) - len(lo)) <= 1, (p, its[p], len(lo))
        if int(its[p]) == len(lo):
            for name, got in (("by", by[p]), ("cx", cx[p])):
                tol = max(1e-7 * max(1.0, abs(lo[-1][name])), 10 * spread[name])
                assert abs(got - lo[-1][name]) <= tol, (p, name, got, lo[-1][name], spread[name])
        assert np.abs(y[p] - yo).max() <= 1e-6 * max(1.0, np.abs(yo).max()), p


def equality_problems(case, count, seed0):
    shape, eqs = CASES[case]
    kw = SHAPES[shape]
    return kw["m"], [small_multicone_equality_problem(seed0 + p, equalities=eqs, **kw) for p in range(count)]


@pytest.mark.parametrize("case,count", [("tiny_2rows", 7), ("mixed_two_blocks", 9), ("c3_8rows", 4)])
def test_batch_with_equalities_matches_oracle_per_program(libs, case, count):
    O, D = libs
    m, problems = equality_problems(case, count, 1000)
    cfg_kw = dict(prepare_dual_variables=1)
    batch = Batch(D, [make_program(D, m, cones) for cones, _ in problems])
    solved, y = batch.maximize(np.stack([pb for _, pb in problems]), D.default_config(**cfg_kw))
    its, by, cx, _ = batch.results()
    check_against_oracle(O, m, problems, solved, y, its, by, cx, cfg_kw)
    assert solved.all()
    for p, (cones, _) in enumerate(problems):  # the equalities hold at the solution
        for kind, A, (b_eq, v) in (c for c in cones if c[0] == "eq"):
            yv = y[p] if v is None else y[p][v]
            assert np.abs(A @ yv - b_eq).max() <= 1e-6 * max(1.0, np.abs(b_eq).max())
    assert batch.milliseconds() > 0 and len(batch.step_milliseconds()) == its.max()


def lp_with_equalities(seed, m=6, ineq=10, eq=3):
    """lb <= A y <= ub with both sides strictly feasible: two-sided rows around A y0 (one with an infinite upper
    bound) and `eq` rows with lb == ub = A y0, which CONEX_AddLinearInequalities turns into an equality block."""
    rng = np.random.Generator(np.random.PCG64(seed))
    A = rng.uniform(-1.0, 1.0, size=(ineq + eq, m))
    y0 = 0.1 * rng.uniform(-1.0, 1.0, size=m)
    center = A @ y0
    width = rng.uniform(0.5, 1.5, size=ineq + eq)
    lb, ub = center - width, center + width
    ub[1] = 1e9
    lb[ineq:] = center[ineq:]
    ub[ineq:] = center[ineq:]
    return A, lb, ub, rng.uniform(-1.0, 1.0, size=m)


def test_batch_lp_with_equalities_from_linear_inequalities(libs):
    O, D = libs
    m, cfg_kw = 6, dict(prepare_dual_variables=1)
    data = [lp_with_equalities(50 + p) for p in range(6)]

    def build(L, A, lb, ub):
        P = L.program(m)
        P.add_linear_inequalities(A, lb, ub)
        return P

    programs = [build(D, A, lb, ub) for A, lb, ub, _ in data]
    assert programs[0].kkt_size() == m + 3
    batch = Batch(D, programs)
    b = np.stack([bb for *_, bb in data])
    solved, y = batch.maximize(b, D.default_config(**cfg_kw))
    its, by, cx, _ = batch.results()
    for p, (A, lb, ub, bb) in enumerate(data):
        P = build(O, A, lb, ub)
        so, yo = P.maximize(bb, O.default_config(**cfg_kw))
        lo = P.iteration_log()
        assert solved[p] == so == 1, p
        assert abs(int(its[p]) - len(lo)) <= 1, (p, its[p], len(lo))
        if int(its[p]) == len(lo):
            assert abs(by[p] - lo[-1]["by"]) <= 1e-7 * max(1.0, abs(lo[-1]["by"])), p
        assert np.abs(y[p] - yo).max() <= 1e-6 * max(1.0, np.abs(yo).max()), p
        assert np.abs(A[10:] @ y[p] - lb[10:]).max() <= 1e-6


def test_batch_with_equalities_matches_single_program_device_path(libs):
    """The same programs through CONEX_Maximize one at a time (dense LDL^T of the KKT system) and through the batch
    (cxb_small_ldlt): same answers."""
    _, D = libs
    m, problems = equality_problems("mixed_two_blocks", 4, 2000)
    singles = []
    for cones, pb in problems:
        Q = make_program(D, m, cones)
        s, y1 = Q.maximize(pb)
        singles.append((s, y1, Q.iteration_log()))
    batch = Batch(D, [make_program(D, m, cones) for cones, _ in problems])
    solved, y = batch.maximize(np.stack([pb for _, pb in problems]))
    its, by, cx, _ = batch.results()
    for p, (s1, y1, log) in enumerate(singles):
        assert solved[p] == s1 and abs(int(its[p]) - len(log)) <= 1
        assert np.abs(y[p] - y1).max() <= 1e-6 * max(1.0, np.abs(y1).max())
        if int(its[p]) == len(log):
            assert abs(by[p] - log[-1]["by"]) <= 1e-7 * max(1.0, abs(by[p]))


def test_programs_with_equalities_finish_at_different_iterations(libs):
    """Masking: programs that terminate early must not be touched by later factorisations and solves."""
    O, D = libs
    m, problems = equality_problems("tiny_2rows", 12, 3000)
    for p in range(12):
        problems[p] = (problems[p][0], problems[p][1] * (1.0 + 3.0 * (p % 4)))
    batch = Batch(D, [make_program(D, m, cones) for cones, _ in problems])
    solved, y = batch.maximize(np.stack([pb for _, pb in problems]))
    its, _, _, _ = batch.results()
    ref_its = []
    for p, (cones, pb) in enumerate(problems):
        P = make_program(O, m, cones)
        so, yo = P.maximize(pb)
        ref_its.append(len(P.iteration_log()))
        assert solved[p] == so
        assert np.abs(y[p] - yo).max() <= 1e-6 * max(1.0, np.abs(yo).max())
    assert len(set(ref_its)) > 1
    assert np.abs(its - np.array(ref_its)).max() <= 1


def test_batch_with_equalities_dual_variables(libs):
    O, D = libs
    m, problems = equality_problems("mixed_two_blocks", 3, 4000)
    cfg_kw = dict(prepare_dual_variables=1)
    batch = Batch(D, [make_program(D, m, cones) for cones, _ in problems])
    batch.maximize(np.stack([pb for _, pb in problems]), D.default_config(**cfg_kw))
    L = D.lib
    for p, (cones, pb) in enumerate(problems):
        P = make_program(O, m, cones)
        P.maximize(pb, O.default_config(**cfg_kw))
        for ci, (kind, A, c) in enumerate(cones):
            if kind == "eq":
                # no dual variable (equality_constraint.h:9-18): size 0, nothing written
                x = np.full(4, 7.0)
                assert L.CONEXB200_BatchGetDualVariable(batch.h, p, ci, dptr(x)) == 0
                assert (x == 7.0).all()
                continue
            if kind == "soc":
                continue  # the reference's SOC dual variable is an unset dummy (workspace_soc.h:44)
            xo = P.dual_variable(ci)
            xd = batch.dual_variable(p, ci, xo.size).reshape(xo.shape, order="F")
            assert np.abs(xo - xd).max() <= 1e-5 * max(1.0, np.abs(xo).max()), (p, ci)


def create_batch(D, programs):
    L = D.lib
    L.CONEXB200_CreateBatch.restype = C.c_void_p
    L.CONEXB200_CreateBatch.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    handles = (C.c_void_p * len(programs))(*[q.h for q in programs])
    return L.CONEXB200_CreateBatch(handles, len(programs))


@pytest.mark.parametrize("other", [((3, None, None),),                       # more rows
                                   ((2, [0, 1, 2], None),),                 # a variable subset
                                   ((2, None, 0),),                         # another position among the cones
                                   ((2, None, None), (1, [3], None))])      # another number of blocks
def test_batch_rejects_mismatched_equality_structure(libs, other):
    _, D = libs
    kw = SHAPES["tiny"]
    ca, _ = small_multicone_equality_problem(1, equalities=((2, None, None),), **kw)
    cb, _ = small_multicone_equality_problem(2, equalities=other, **kw)
    assert not create_batch(D, [make_program(D, kw["m"], ca), make_program(D, kw["m"], cb)])
    # the same structure is accepted
    cc, _ = small_multicone_equality_problem(3, equalities=((2, None, None),), **kw)
    h = create_batch(D, [make_program(D, kw["m"], ca), make_program(D, kw["m"], cc)])
    assert h
    D.lib.CONEXB200_DeleteBatch.argtypes = [C.c_void_p]
    D.lib.CONEXB200_DeleteBatch(h)


def test_batch_with_equalities_refuses_iterative_refinement(libs):
    _, D = libs
    m, problems = equality_problems("tiny_2rows", 2, 5000)
    batch = Batch(D, [make_program(D, m, cones) for cones, _ in problems])
    b = np.stack([pb for _, pb in problems])
    with pytest.raises(AssertionError, match="BatchMaximize failed"):
        batch.maximize(b, D.default_config(iterative_refinement_iterations=1))
    solved, _ = batch.maximize(b)  # the batch stays usable
    assert solved.all()


def test_batch_refuses_line_search_on_lp_and_equalities_only(libs):
    _, D = libs
    m = 6
    data = [lp_with_equalities(70 + p) for p in range(2)]
    programs = []
    for A, lb, ub, _ in data:
        P = D.program(m)
        P.add_linear_inequalities(A, lb, ub)
        programs.append(P)
    batch = Batch(D, programs)
    with pytest.raises(AssertionError, match="BatchMaximize failed"):
        batch.maximize(np.stack([bb for *_, bb in data]), D.default_config(enable_line_search=1))
