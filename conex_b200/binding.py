"""ctypes binding of the CONEX_* C ABI and of the cxb_* device layer, shared by bench.py,
__graft_entry__.smoke() and the tests.

Two shared libraries speak the same `CONEX_*` C ABI (include/conex.h, the reference's
interfaces/conex.h):

* the CPU oracle   oracle/_build/libconex_oracle.so  (test infrastructure), and
* the product      conex_b200/lib/libconex_b200.so   (hand-written sm_100a CUDA).

`ConexLib` wraps either so that a parity test reads like the reference's own tests
(conex/test/test_sdp.cc, interfaces/python/test/run_tests.py): build a program, add constraints,
Maximize, inspect y / dual variables / iteration stats.
"""
import ctypes as C
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PRODUCT_SO = os.path.join(ROOT, "conex_b200", "lib", "libconex_b200.so")

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)


class SolverConfiguration(C.Structure):
    """Mirror of CONEX_SolverConfiguration (include/conex.h; reference conex.h:10-30)."""

    _fields_ = [
        ("prepare_dual_variables", C.c_int),
        ("initialization_mode", C.c_int),
        ("inv_sqrt_mu_max", C.c_double),
        ("minimum_mu", C.c_double),
        ("maximum_mu", C.c_double),
        ("divergence_upper_bound", C.c_double),
        ("enable_line_search", C.c_int),
        ("dinf_upper_bound", C.c_double),
        ("final_centering_steps", C.c_int),
        ("final_centering_tolerance", C.c_double),
        ("initial_centering_steps_warmstart", C.c_int),
        ("initial_centering_steps_coldstart", C.c_int),
        ("warmstart_abort_threshold", C.c_double),
        ("max_iterations", C.c_int),
        ("iterative_refinement_iterations", C.c_int),
        ("infeasibility_threshold", C.c_double),
        ("kkt_error_tolerance", C.c_double),
        ("enable_rescaling", C.c_int),
        ("kkt_solver", C.c_int),
    ]


class IterationStats(C.Structure):
    _fields_ = [("mu", C.c_double), ("iteration_number", C.c_int)]


def dptr(a):
    return a.ctypes.data_as(c_double_p)


def fmat(a):
    """Column-major float64 copy (what the C ABI expects)."""
    return np.asfortranarray(np.array(a, dtype=np.float64))


def pack_matrices(mats):
    """m symmetric n x n matrices -> one contiguous buffer of m column-major blocks."""
    return np.ascontiguousarray(np.stack([np.asfortranarray(M).ravel(order="F") for M in mats]))


class ConexLib:
    """A loaded CONEX_* library (oracle or product)."""

    def __init__(self, path, kind):
        self.kind = kind  # "oracle" | "b200"
        self.path = path
        self.lib = C.CDLL(path)
        L = self.lib
        L.CONEX_CreateConeProgram.restype = C.c_void_p
        L.CONEX_DeleteConeProgram.argtypes = [C.c_void_p]
        L.CONEX_SetNumberOfVariables.argtypes = [C.c_void_p, C.c_int]
        L.CONEX_AddDenseLMIConstraint.argtypes = [C.c_void_p, c_double_p, C.c_int, C.c_int, C.c_int,
                                                  c_double_p, C.c_int, C.c_int]
        L.CONEX_AddSparseLMIConstraint.argtypes = [C.c_void_p, c_double_p, C.c_int, C.c_int, C.c_int,
                                                   c_double_p, C.c_int, C.c_int,
                                                   C.POINTER(C.c_long), C.c_int]
        L.CONEX_AddDenseLinearConstraint.argtypes = [C.c_void_p, c_double_p, C.c_int, C.c_int,
                                                     c_double_p, C.c_int]
        L.CONEX_Maximize.argtypes = [C.c_void_p, c_double_p, C.c_int,
                                     C.POINTER(SolverConfiguration), c_double_p, C.c_int]
        L.CONEX_GetDualVariable.argtypes = [C.c_void_p, C.c_int, c_double_p, C.c_int, C.c_int]
        L.CONEX_GetDualVariableSize.argtypes = [C.c_void_p, C.c_int]
        L.CONEX_SetDefaultOptions.argtypes = [C.POINTER(SolverConfiguration)]
        L.CONEX_GetIterationStats.argtypes = [C.c_void_p, C.POINTER(IterationStats), C.c_int]
        L.CONEX_AddLinearInequalities.argtypes = [C.c_void_p, c_double_p, C.c_int, C.c_int, c_double_p,
                                                  C.c_int, c_double_p, C.c_int]
        L.CONEX_NewLorentzConeConstraint.argtypes = [C.c_void_p, C.c_int, c_int_p]
        L.CONEX_NewLinearInequality.argtypes = [C.c_void_p, C.c_int, c_int_p]
        L.CONEX_NewLinearMatrixInequality.argtypes = [C.c_void_p, C.c_int, C.c_int, c_int_p]
        L.CONEX_UpdateLinearOperator.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_int,
                                                 C.c_int, C.c_int]
        L.CONEX_UpdateAffineTerm.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int]
        self.ext = "ORACLE" if kind == "oracle" else "CONEXB200"
        for name, args, res in [
            ("FeasibleObjective", [C.c_void_p, c_double_p], None),
            ("GetStatus", [C.c_void_p, c_int_p], None),
            ("GetIterationLog", [C.c_void_p, C.c_int, c_double_p], C.c_int),
            ("GetPhaseSeconds", [C.c_void_p, c_double_p], None),
            ("AssembleNewtonSystem", [C.c_void_p, C.c_int, c_double_p, c_double_p, c_double_p,
                                      c_double_p], None),
            ("AddSocConstraint", [C.c_void_p, C.c_int, C.c_int, c_double_p, c_double_p], C.c_int),
            ("AddEqualityConstraint", [C.c_void_p, C.c_int, C.c_int, c_double_p, c_double_p,
                                       C.POINTER(C.c_long)], C.c_int),
            ("SizeOfKKTSystem", [C.c_void_p], C.c_int),
        ]:
            f = getattr(L, f"{self.ext}_{name}")
            f.argtypes = args
            f.restype = res
        if kind != "oracle":  # cones on variable subsets: product library only
            L.CONEXB200_AddSparseLinearConstraint.argtypes = [C.c_void_p, c_double_p, C.c_int, C.c_int, c_double_p,
                                                              C.POINTER(C.c_long)]
            L.CONEXB200_AddSparseSocConstraint.argtypes = [C.c_void_p, C.c_int, C.c_int, c_double_p, c_double_p,
                                                           C.POINTER(C.c_long)]

    def fn(self, name):
        return getattr(self.lib, f"{self.ext}_{name}")

    def default_config(self, **kw):
        cfg = SolverConfiguration()
        self.lib.CONEX_SetDefaultOptions(C.byref(cfg))
        for k, v in kw.items():
            setattr(cfg, k, v)
        return cfg

    def program(self, m=0):
        return Program(self, m)

    def program_on_memory_of(self, other, m=0):
        """`Program prog2(m, &prog.memory_)` of the reference (cone_program.h:106-109): product library only."""
        f = self.lib.CONEXB200_CreateConeProgramOnMemoryOf
        f.restype = C.c_void_p
        f.argtypes = [C.c_void_p]
        handle = f(other.h)
        assert handle, "CONEXB200_CreateConeProgramOnMemoryOf failed"
        return Program(self, m, handle=handle)


class Program:
    """Mirror of the reference's Python `Conex` class (interfaces/python/ConexProgram.py:58-277),
    reduced to the hot path."""

    def __init__(self, lib, m=0, handle=None):
        self.L = lib
        self.h = C.c_void_p(handle if handle is not None else lib.lib.CONEX_CreateConeProgram())
        self.m = 0
        self.cone_shapes = []
        if m > 0:
            assert lib.lib.CONEX_SetNumberOfVariables(self.h, m) == 0
            self.m = m
        self._keep = []

    def __del__(self):
        try:
            self.L.lib.CONEX_DeleteConeProgram(self.h)
        except Exception:
            pass

    def add_dense_lmi(self, mats, Cmat, variables=None):
        n = Cmat.shape[0]
        A = pack_matrices(mats)
        Cf = fmat(Cmat)
        m = len(mats)
        if variables is None:
            cid = self.L.lib.CONEX_AddDenseLMIConstraint(self.h, dptr(A), n, n, m, dptr(Cf), n, n)
            if self.m == 0:
                self.m = m
        else:
            v = (C.c_long * m)(*variables)
            cid = self.L.lib.CONEX_AddSparseLMIConstraint(self.h, dptr(A), n, n, m, dptr(Cf), n, n, v, m)
        self.cone_shapes.append((n, n))
        return cid

    def add_dense_lmi_packed(self, A, Cf, n, m):
        """A: contiguous (m, n*n) buffer of column-major blocks; Cf: column-major n x n."""
        cid = self.L.lib.CONEX_AddDenseLMIConstraint(self.h, dptr(A), n, n, m, dptr(Cf), n, n)
        if self.m == 0:
            self.m = m
        self.cone_shapes.append((n, n))
        return cid

    def add_linear(self, A, c, variables=None):
        """c - A y >= 0. variables: the list of variables A's columns act on (CONEXB200_AddSparseLinearConstraint,
        product library only; the program's number of variables must be set); None = all of them."""
        Af = fmat(A)
        cf = np.ascontiguousarray(np.array(c, dtype=np.float64).ravel())
        if variables is not None:
            v = (C.c_long * len(variables))(*variables)
            cid = self.L.lib.CONEXB200_AddSparseLinearConstraint(self.h, dptr(Af), Af.shape[0], Af.shape[1],
                                                                 dptr(cf), v)
            if cid >= 0:
                self.cone_shapes.append((Af.shape[0], 1))
            return cid
        cid = self.L.lib.CONEX_AddDenseLinearConstraint(self.h, dptr(Af), Af.shape[0], Af.shape[1],
                                                        dptr(cf), Af.shape[0])
        if self.m == 0:
            self.m = Af.shape[1]
        self.cone_shapes.append((Af.shape[0], 1))
        return cid

    def add_soc(self, A, c, incremental=False, variables=None):
        """c - A y in the Lorentz cone of order n+1 (A is (n+1) x m). incremental=True goes through
        CONEX_NewLorentzConeConstraint + CONEX_UpdateLinearOperator / CONEX_UpdateAffineTerm like
        interfaces/python/test/run_tests.py:23-34; otherwise through the SOCConstraint(A, c)
        constructor the reference's C++ tests use (conex/test/test_socp.cc:41-46). variables: the list of
        variables A's columns act on (CONEXB200_AddSparseSocConstraint, product library only; the program's
        number of variables must be set); None = all of them."""
        Af = fmat(A)
        cf = np.ascontiguousarray(np.array(c, dtype=np.float64).ravel())
        order = Af.shape[0] - 1
        if variables is not None:
            assert not incremental
            v = (C.c_long * len(variables))(*variables)
            cid = self.L.lib.CONEXB200_AddSparseSocConstraint(self.h, order, Af.shape[1], dptr(Af), dptr(cf), v)
            if cid >= 0:
                self.cone_shapes.append((order + 1, 1))
            return cid
        if self.m == 0:
            assert self.L.lib.CONEX_SetNumberOfVariables(self.h, Af.shape[1]) == 0
            self.m = Af.shape[1]
        if incremental:
            cid = C.c_int(-1)
            assert self.L.lib.CONEX_NewLorentzConeConstraint(self.h, order, C.byref(cid)) == 0
            cid = cid.value
            for r in range(order + 1):
                assert self.L.lib.CONEX_UpdateAffineTerm(self.h, cid, float(cf[r]), r, 0, 0) == 0
                for v in range(Af.shape[1]):
                    assert self.L.lib.CONEX_UpdateLinearOperator(self.h, cid, float(Af[r, v]), v, r, 0, 0) == 0
        else:
            cid = self.L.fn("AddSocConstraint")(self.h, order, Af.shape[1], dptr(Af), dptr(cf))
        self.cone_shapes.append((order + 1, 1))
        return cid

    def add_hermitian_lmi(self, mats, Cmat):
        """The incremental real LMI (HermitianPsdConstraint<Real>): CONEX_NewLinearMatrixInequality +
        CONEX_UpdateLinearOperator / CONEX_UpdateAffineTerm on the lower triangle, as
        interfaces/python/test/run_tests.py:5-21 does."""
        n = Cmat.shape[0]
        if self.m == 0:
            assert self.L.lib.CONEX_SetNumberOfVariables(self.h, len(mats)) == 0
            self.m = len(mats)
        cid = C.c_int(-1)
        assert self.L.lib.CONEX_NewLinearMatrixInequality(self.h, n, 1, C.byref(cid)) == 0
        for r in range(n):
            for c in range(r + 1):
                if Cmat[r, c] != 0:
                    assert self.L.lib.CONEX_UpdateAffineTerm(self.h, cid.value, float(Cmat[r, c]), r, c, 0) == 0
                for v, M in enumerate(mats):
                    if M[r, c] != 0:
                        assert self.L.lib.CONEX_UpdateLinearOperator(self.h, cid.value, float(M[r, c]), v, r, c, 0) == 0
        self.cone_shapes.append((n, n))
        return cid.value

    def add_linear_incremental(self, A, c):
        """CONEX_NewLinearInequality + per-entry updates (interfaces/conex.cc:318-329)."""
        Af = fmat(A)
        cf = np.array(c, dtype=np.float64).ravel()
        cid = C.c_int(-1)
        assert self.L.lib.CONEX_NewLinearInequality(self.h, Af.shape[0], C.byref(cid)) == 0
        for r in range(Af.shape[0]):
            assert self.L.lib.CONEX_UpdateAffineTerm(self.h, cid.value, float(cf[r]), r, 0, 0) == 0
            for v in range(Af.shape[1]):
                assert self.L.lib.CONEX_UpdateLinearOperator(self.h, cid.value, float(Af[r, v]), v, r, 0, 0) == 0
        self.cone_shapes.append((Af.shape[0], 1))
        return cid.value

    def add_linear_inequalities(self, A, lb, ub):
        """lb <= A y <= ub (CONEX_AddLinearInequalities, interfaces/conex.cc:190-215): equal bounds
        become equality constraints, finite ones scaled inequality rows."""
        Af = fmat(A)
        lbf = np.ascontiguousarray(np.array(lb, dtype=np.float64).ravel())
        ubf = np.ascontiguousarray(np.array(ub, dtype=np.float64).ravel())
        r = self.L.lib.CONEX_AddLinearInequalities(self.h, dptr(Af), Af.shape[0], Af.shape[1], dptr(lbf),
                                                   len(lbf), dptr(ubf), len(ubf))
        eq = lbf == ubf
        nin = int(((ubf < 1e8) & ~eq).sum() + ((lbf > -1e8) & ~eq).sum())
        if nin:
            self.cone_shapes.append((nin, 1))
        if eq.any():
            self.cone_shapes.append((0, 0))
        return r

    def add_equality(self, A, b, variables=None):
        """A y[variables] = b (Program::AddConstraint(EqualityConstraints{A, b}[, vars]))."""
        Af = fmat(A)
        bf = np.ascontiguousarray(np.array(b, dtype=np.float64).ravel())
        v = None if variables is None else (C.c_long * len(variables))(*variables)
        cid = self.L.fn("AddEqualityConstraint")(self.h, Af.shape[0], Af.shape[1], dptr(Af), dptr(bf), v)
        assert cid >= 0
        self.cone_shapes.append((0, 0))
        return cid

    def dense_lmi_storage(self, n, m, world=1, rank=0):
        """Library-owned device storage of a dense LMI block (CONEXB200_NewDenseLMIConstraintStorage):
        returns torch views (no copy) `A` (row_count x n*n, one column-major n x n block per row) and
        `Cm` (n x n) to be filled in place, and this rank's row range of the m constraint matrices."""
        from .workloads import device_view
        L = self.L.lib
        b, c = C.c_int(), C.c_int()
        L.CONEXB200_ShardRange(m, world, rank, C.byref(b), C.byref(c))
        pA, pC = C.c_void_p(), C.c_void_p()
        cid = L.CONEXB200_NewDenseLMIConstraintStorage(self.h, n, m, C.byref(pA), C.byref(pC))
        assert cid >= 0, "allocation of the constraint matrices failed"
        self.m = m
        self.cone_shapes.append((n, n))
        A = device_view(pA.value, c.value * n * n).view(c.value, n * n)
        Cm = device_view(pC.value, n * n).view(n, n)
        return A, Cm, b.value, c.value

    def add_entry_lmi(self, n, entries, Cmat):
        """An LMI given entry by entry (CONEX_NewLinearMatrixInequality + CONEX_UpdateLinearOperator /
        CONEX_UpdateAffineTerm): entries = [(variable, row, col, value)] on the lower triangle."""
        L = self.L.lib
        cid = C.c_int(-1)
        assert L.CONEX_NewLinearMatrixInequality(self.h, n, 1, C.byref(cid)) == 0
        for (v, r, c, val) in entries:
            assert L.CONEX_UpdateLinearOperator(self.h, cid.value, float(val), v, r, c, 0) == 0
        rr, cc = np.nonzero(np.tril(Cmat))
        for r, c in zip(rr.tolist(), cc.tolist()):
            assert L.CONEX_UpdateAffineTerm(self.h, cid.value, float(Cmat[r, c]), r, c, 0) == 0
        self.cone_shapes.append((n, n))
        return cid.value

    def kkt_size(self):
        return self.L.fn("SizeOfKKTSystem")(self.h)

    def feasible_objective(self):
        b = np.zeros(self.m)
        self.L.fn("FeasibleObjective")(self.h, dptr(b))
        return b

    def maximize(self, b, cfg=None):
        if cfg is None:
            cfg = self.L.default_config()
        b = np.ascontiguousarray(np.array(b, dtype=np.float64).ravel())
        y = np.zeros(self.m)
        solved = self.L.lib.CONEX_Maximize(self.h, dptr(b), self.m, C.byref(cfg), dptr(y), self.m)
        return solved, y

    def dual_variable(self, i):
        r, c = self.cone_shapes[i]
        assert self.L.lib.CONEX_GetDualVariableSize(self.h, i) == r * c
        x = np.zeros(r * c)
        self.L.lib.CONEX_GetDualVariable(self.h, i, dptr(x), r, c)
        return x.reshape((r, c), order="F")

    def status(self):
        out = (C.c_int * 4)()
        self.L.fn("GetStatus")(self.h, out)
        return dict(solved=out[0], num_iterations=out[1], primal_infeasible=out[2],
                    dual_infeasible=out[3])

    def iteration_log(self):
        """List of dicts {inv_sqrt_mu, mu, d_2, d_inf, by, cx, kkt_error, step_size}."""
        keys = ["inv_sqrt_mu", "mu", "d_2", "d_inf", "by", "cx", "kkt_error", "step_size"]
        rows = []
        buf = np.zeros(8)
        i = 0
        while self.L.fn("GetIterationLog")(self.h, i, dptr(buf)):
            rows.append(dict(zip(keys, buf.tolist())))
            i += 1
        return rows

    def iteration_stats(self, it):
        s = IterationStats()
        s.mu = float("nan")
        s.iteration_number = -12345
        self.L.lib.CONEX_GetIterationStats(self.h, C.byref(s), it)
        return s.mu, s.iteration_number

    def phase_seconds(self):
        buf = np.zeros(5)
        self.L.fn("GetPhaseSeconds")(self.h, dptr(buf))
        return dict(zip(["assemble", "factor", "solve", "update", "mu"], buf.tolist()))

    def newton_system(self, coldstart=True):
        m = self.kkt_size()
        H = np.zeros((m, m), order="F")
        AW = np.zeros(m)
        AQc = np.zeros(m)
        sc = np.zeros(2)
        self.L.fn("AssembleNewtonSystem")(self.h, 1 if coldstart else 0, dptr(H), dptr(AW), dptr(AQc),
                                          dptr(sc))
        return np.tril(H), AW, AQc, sc


class Batch:
    """CONEXB200_CreateBatch / BatchMaximize on a list of harness Programs (product library only)."""

    def __init__(self, lib, programs):
        self.L = lib
        L = lib.lib
        L.CONEXB200_CreateBatch.restype = C.c_void_p
        L.CONEXB200_CreateBatch.argtypes = [C.POINTER(C.c_void_p), C.c_int]
        L.CONEXB200_DeleteBatch.argtypes = [C.c_void_p]
        L.CONEXB200_BatchMaximize.argtypes = [C.c_void_p, c_double_p, C.POINTER(SolverConfiguration), c_double_p,
                                              c_int_p]
        L.CONEXB200_BatchGetResults.argtypes = [C.c_void_p, c_int_p, c_double_p, c_double_p, c_double_p]
        L.CONEXB200_BatchMilliseconds.restype = C.c_double
        L.CONEXB200_BatchMilliseconds.argtypes = [C.c_void_p]
        L.CONEXB200_BatchStepMilliseconds.argtypes = [C.c_void_p, c_double_p, C.c_int]
        L.CONEXB200_BatchGetDualVariable.argtypes = [C.c_void_p, C.c_int, C.c_int, c_double_p]
        L.CONEXB200_BatchUpdateConstraintData.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, c_double_p]
        L.CONEXB200_BatchConstraintDataShape.argtypes = [C.c_void_p, C.c_int, c_int_p, c_int_p]
        self.count = len(programs)
        self.m = programs[0].m
        handles = (C.c_void_p * self.count)(*[p.h for p in programs])
        self.h = C.c_void_p(L.CONEXB200_CreateBatch(handles, self.count))
        assert self.h.value, "CONEXB200_CreateBatch failed"

    def __del__(self):
        try:
            self.L.lib.CONEXB200_DeleteBatch(self.h)
        except Exception:
            pass

    def maximize(self, b, cfg=None):
        """b: (count, m). Returns (solved (count,), y (count, m))."""
        if cfg is None:
            cfg = self.L.default_config()
        b = np.ascontiguousarray(np.asarray(b, dtype=np.float64))
        y = np.zeros((self.count, self.m))
        solved = (C.c_int * self.count)()
        rc = self.L.lib.CONEXB200_BatchMaximize(self.h, dptr(b), C.byref(cfg), dptr(y), solved)
        assert rc >= 0, "CONEXB200_BatchMaximize failed"
        return np.array(list(solved)), y

    def update(self, constraint, first, data):
        """CONEXB200_BatchUpdateConstraintData: data (count, rows, ncols) replaces columns [first, first + ncols) of
        constraint `constraint` in every program."""
        data = np.asarray(data, dtype=np.float64)
        rows, columns = C.c_int(), C.c_int()
        assert self.L.lib.CONEXB200_BatchConstraintDataShape(self.h, constraint, C.byref(rows), C.byref(columns)) == 0
        assert data.ndim == 3 and data.shape[:2] == (self.count, rows.value), (data.shape, rows.value)
        blocks = np.ascontiguousarray(data.transpose(0, 2, 1))  # program p: rows x ncols column-major
        rc = self.L.lib.CONEXB200_BatchUpdateConstraintData(self.h, constraint, first, data.shape[2], dptr(blocks))
        assert rc == 0, "CONEXB200_BatchUpdateConstraintData failed"

    def results(self):
        it = (C.c_int * self.count)()
        by, cx, k = np.zeros(self.count), np.zeros(self.count), np.zeros(self.count)
        self.L.lib.CONEXB200_BatchGetResults(self.h, it, dptr(by), dptr(cx), dptr(k))
        return np.array(list(it)), by, cx, k

    def milliseconds(self):
        return self.L.lib.CONEXB200_BatchMilliseconds(self.h)

    def step_milliseconds(self):
        buf = np.zeros(256)
        n = self.L.lib.CONEXB200_BatchStepMilliseconds(self.h, dptr(buf), 256)
        return buf[:n].copy()

    def dual_variable(self, p, cone, size):
        x = np.zeros(size)
        assert self.L.lib.CONEXB200_BatchGetDualVariable(self.h, p, cone, dptr(x)) == size
        return x


# ----------------------------------------------------------------------------------------------
# cxb_* device layer (include/conex_b200_device.h). torch is used only to own device memory: a
# column-major r x c matrix is a torch tensor of shape (c, r), so `tensor.data_ptr()` is exactly the
# `double*` the C ABI expects.
# ----------------------------------------------------------------------------------------------
vp = C.c_void_p
_dev = None


def product():
    """The product library as a CONEX_* speaker plus its cxb_* kernels. Fails loudly if missing."""
    global _dev
    if _dev is None:
        if not os.path.exists(PRODUCT_SO):
            raise RuntimeError(f"{PRODUCT_SO} is missing: run `python -c 'import __graft_entry__ as g; "
                               "g.build()'` — conex-b200 has no CPU fallback")
        _dev = ConexLib(PRODUCT_SO, "b200")
        L = _dev.lib
        L.cxb_dgemm.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, vp, C.c_long,
                                C.c_long, vp, C.c_long, C.c_long, C.c_double, vp, C.c_long, C.c_long,
                                C.c_int, C.c_int]
        L.cxb_dgemm_ex.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_double, vp, C.c_long, C.c_long, vp, C.c_long, C.c_long, C.c_double,
                                   vp, C.c_long, C.c_long, C.c_int, C.c_int, C.c_int, C.c_int]
        L.cxb_dgemm_bulk.argtypes = [vp, C.c_int, C.c_int, C.c_int, vp, C.c_long, C.c_long, vp, C.c_long, C.c_long, vp,
                                     C.c_long, C.c_long, C.c_int, C.c_int]
        L.cxb_set_default_gemm_config.argtypes = [C.c_int]
        L.cxb_set_default_gemm_config.restype = None
        L.cxb_schur_dense_lmi.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp, C.c_int, vp, C.c_long]
        L.cxb_schur_dense_lmi_streamed.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp, C.c_int, vp, C.c_long]
        L.CONEXB200_SetAssemblyMode.argtypes = [vp, C.c_int]
        L.CONEXB200_SetAssemblyMode.restype = None
        L.cxb_potrf_lower.argtypes = [vp, C.c_int, vp, C.c_long, vp, vp]
        L.cxb_potrs_lower.argtypes = [vp, C.c_int, vp, C.c_long, vp, C.c_long, C.c_int]
        L.cxb_gemv_n.argtypes = [vp, C.c_long, C.c_int, vp, vp, vp]
        L.cxb_lanczos_worksize.argtypes = [C.c_int]
        L.cxb_lanczos_worksize.restype = C.c_size_t
        L.cxb_lanczos_two_sided.argtypes = [vp, C.c_int, vp, vp, vp, vp, C.c_int, vp, vp, vp, vp]
        L.cxb_ws_reductions.argtypes = [vp, C.c_int, vp, vp]
        L.cxb_geodesic_worksize.argtypes = [C.c_int]
        L.cxb_geodesic_worksize.restype = C.c_size_t
        L.cxb_geodesic_update.argtypes = [vp, C.c_int, vp, vp, C.c_double, C.c_double, vp, vp, vp]
        L.cxb_pade_expm.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp]
        L.cxb_lu_solve.argtypes = [vp, C.c_int, vp, C.c_long, C.c_int, vp, C.c_long, vp, vp]
        L.cxb_set_identity.argtypes = [vp, C.c_int, vp]
        L.cxb_dot.argtypes = [vp, C.c_long, vp, vp, vp]
        L.cxb_axpbypcz.argtypes = [vp, C.c_long, C.c_double, vp, C.c_double, vp, C.c_double, vp]
        L.cxb_copy_strided.argtypes = [vp, C.c_long, vp, C.c_long, vp, C.c_long]
        L.cxb_scatter_add_lower.argtypes = [vp, C.c_int, vp, C.c_long, vp, vp, C.c_long]
        L.cxb_fill.argtypes = [vp, C.c_long, C.c_double, vp]
        L.cxb_scatter_add_vec.argtypes = [vp, C.c_int, vp, vp, vp]
        L.cxb_gather_vec.argtypes = [vp, C.c_int, vp, vp, vp]
        L.cxb_affine_update.argtypes = [vp, C.c_int, vp, vp, C.c_double]
        L.CONEXB200_AddDenseLMIConstraintDevice.argtypes = [vp, vp, C.c_int, C.c_int, vp]
        L.CONEXB200_AddDenseLMIConstraintShard.argtypes = [vp, vp, C.c_int, C.c_int, vp]
        L.CONEXB200_NewDenseLMIConstraintStorage.argtypes = [vp, C.c_int, C.c_int, C.POINTER(vp), C.POINTER(vp)]
        L.CONEXB200_CommGetUniqueId.argtypes = [C.c_char_p]
        L.CONEXB200_CommInitRank.argtypes = [C.c_int, C.c_int, C.c_char_p]
        L.CONEXB200_CommDestroy.restype = None
        L.CONEXB200_ShardRange.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.CONEXB200_ShardRange.restype = None
        L.CONEXB200_GetIterationMilliseconds.argtypes = [vp, C.c_int, C.POINTER(C.c_double)]
        L.CONEXB200_SetTiming.argtypes = [vp, C.c_int]
        L.CONEXB200_GetIterationPhaseMilliseconds.argtypes = [vp, C.c_int, C.POINTER(C.c_double)]
        L.CONEXB200_DivergenceUpperBoundInverse.argtypes = [C.c_double] * 6
        L.CONEXB200_DivergenceUpperBoundInverse.restype = C.c_double
        L.CONEXB200_TridiagonalExtremes.argtypes = [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.CONEXB200_LaunchCount.restype = C.c_long
        L.CONEXB200_SetCollective.argtypes = [vp, C.c_int]
        L.CONEXB200_SetCollective.restype = None
        L.CONEXB200_SetDistributedCholesky.argtypes = [C.c_int, C.c_int]
        L.CONEXB200_SetDistributedCholesky.restype = None
        L.CONEXB200_DistributedPotrf.argtypes = [C.c_int, vp, C.c_long, C.c_int, C.POINTER(C.c_int)]
        L.cxb_potrf_begin.argtypes = [vp, vp]
        L.cxb_potrf_panel.argtypes = [vp, C.c_int, C.c_int, C.c_int, vp, C.c_long, vp]
    return _dev


def to_dev(a):
    """numpy (r x c or 1-D) -> torch cuda tensor whose memory is the column-major matrix."""
    import torch
    a = np.asarray(a, dtype=np.float64)
    if a.ndim == 1:
        return torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return torch.from_numpy(np.ascontiguousarray(a.T)).cuda()


def from_dev(t, rows=None, cols=None):
    import torch
    torch.cuda.synchronize()
    h = t.cpu().numpy()
    if h.ndim == 1 and rows is None:
        return h.copy()
    if rows is not None:
        return h.reshape(-1)[: rows * cols].reshape((cols, rows)).T.copy()
    return h.T.copy()


def dzeros(*shape):
    import torch
    return torch.zeros(*shape, dtype=torch.float64, device="cuda")


def izeros(n):
    import torch
    return torch.zeros(n, dtype=torch.int32, device="cuda")


def ptr(t):
    return C.c_void_p(t.data_ptr())


def init_communicator(dev, rank, world):
    """Rendezvous of the library's NCCL communicator over an initialised torch.distributed group:
    rank 0 creates the unique id, torch broadcasts its 128 bytes, every rank joins."""
    import torch
    import torch.distributed as dist
    L = dev.lib
    buf = C.create_string_buffer(128)
    if rank == 0:
        assert L.CONEXB200_CommGetUniqueId(buf) == 0
    t = torch.tensor(list(buf.raw), dtype=torch.uint8, device="cuda")
    dist.broadcast(t, 0)
    ident = bytes(t.cpu().tolist())
    assert L.CONEXB200_CommInitRank(world, rank, ident) == 0


def shard_range(dev, m, world, rank):
    b, c = C.c_int(), C.c_int()
    dev.lib.CONEXB200_ShardRange(m, world, rank, C.byref(b), C.byref(c))
    return b.value, c.value
