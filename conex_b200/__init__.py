"""conex_b200 — B200-native Newton step of conex's geodesic interior-point method.

The product is the shared library `conex_b200/lib/libconex_b200.so` (CONEX_* C ABI of
include/conex.h over hand-written sm_100a CUDA). This module is the host-side mirror of the
reference's Python front end (interfaces/python/ConexProgram.py:58-277, class `Conex`) over ctypes
instead of SWIG: same method names, same argument meaning, same error behaviour (NameError on a
failed call). There is no CPU fallback: if the library is missing, import fails loudly.
"""
import ctypes as _C
import os as _os

import numpy as _np

_HERE = _os.path.dirname(_os.path.abspath(__file__))
LIBRARY_PATH = _os.path.join(_HERE, "lib", "libconex_b200.so")

if not _os.path.exists(LIBRARY_PATH):
    raise ImportError(
        f"{LIBRARY_PATH} not found. Build it with `make -C {_HERE}` (or __graft_entry__.build()); "
        "conex_b200 has no CPU or PyTorch fallback.")

_lib = _C.CDLL(LIBRARY_PATH)
_dp = _C.POINTER(_C.c_double)


class CONEX_SolverConfiguration(_C.Structure):
    """include/conex.h (reference interfaces/conex.h:10-30)."""
    _fields_ = [
        ("prepare_dual_variables", _C.c_int), ("initialization_mode", _C.c_int),
        ("inv_sqrt_mu_max", _C.c_double), ("minimum_mu", _C.c_double), ("maximum_mu", _C.c_double),
        ("divergence_upper_bound", _C.c_double), ("enable_line_search", _C.c_int),
        ("dinf_upper_bound", _C.c_double), ("final_centering_steps", _C.c_int),
        ("final_centering_tolerance", _C.c_double), ("initial_centering_steps_warmstart", _C.c_int),
        ("initial_centering_steps_coldstart", _C.c_int), ("warmstart_abort_threshold", _C.c_double),
        ("max_iterations", _C.c_int), ("iterative_refinement_iterations", _C.c_int),
        ("infeasibility_threshold", _C.c_double), ("kkt_error_tolerance", _C.c_double),
        ("enable_rescaling", _C.c_int), ("kkt_solver", _C.c_int),
    ]


class CONEX_IterationStats(_C.Structure):
    _fields_ = [("mu", _C.c_double), ("iteration_number", _C.c_int)]


def bind_conex_abi(lib):
    """Declares the argument types of the CONEX_* entry points (include/conex.h) on `lib` — the product,
    or any other library that speaks the same C ABI (the test-suite drives the CPU oracle through this
    very class that way)."""
    lib.CONEX_CreateConeProgram.restype = _C.c_void_p
    lib.CONEX_DeleteConeProgram.argtypes = [_C.c_void_p]
    lib.CONEX_SetNumberOfVariables.argtypes = [_C.c_void_p, _C.c_int]
    lib.CONEX_AddDenseLMIConstraint.argtypes = [_C.c_void_p, _dp, _C.c_int, _C.c_int, _C.c_int, _dp,
                                                 _C.c_int, _C.c_int]
    lib.CONEX_AddSparseLMIConstraint.argtypes = [_C.c_void_p, _dp, _C.c_int, _C.c_int, _C.c_int, _dp,
                                                  _C.c_int, _C.c_int, _C.POINTER(_C.c_long), _C.c_int]
    lib.CONEX_Maximize.argtypes = [_C.c_void_p, _dp, _C.c_int, _C.POINTER(CONEX_SolverConfiguration), _dp,
                                    _C.c_int]
    lib.CONEX_GetDualVariable.argtypes = [_C.c_void_p, _C.c_int, _dp, _C.c_int, _C.c_int]
    lib.CONEX_GetDualVariableSize.argtypes = [_C.c_void_p, _C.c_int]
    lib.CONEX_SetDefaultOptions.argtypes = [_C.POINTER(CONEX_SolverConfiguration)]
    lib.CONEX_GetIterationStats.argtypes = [_C.c_void_p, _C.POINTER(CONEX_IterationStats), _C.c_int]
    _ip = _C.POINTER(_C.c_int)
    lib.CONEX_AddDenseLinearConstraint.argtypes = [_C.c_void_p, _dp, _C.c_int, _C.c_int, _dp, _C.c_int]
    lib.CONEX_AddLinearInequalities.argtypes = [_C.c_void_p, _dp, _C.c_int, _C.c_int, _dp, _C.c_int, _dp, _C.c_int]
    lib.CONEX_NewLinearMatrixInequality.argtypes = [_C.c_void_p, _C.c_int, _C.c_int, _ip]
    lib.CONEX_NewLorentzConeConstraint.argtypes = [_C.c_void_p, _C.c_int, _ip]
    lib.CONEX_NewLinearInequality.argtypes = [_C.c_void_p, _C.c_int, _ip]
    lib.CONEX_UpdateLinearOperator.argtypes = [_C.c_void_p, _C.c_int, _C.c_double, _C.c_int, _C.c_int, _C.c_int,
                                                _C.c_int]
    lib.CONEX_UpdateAffineTerm.argtypes = [_C.c_void_p, _C.c_int, _C.c_double, _C.c_int, _C.c_int, _C.c_int]
    return lib


_ip = _C.POINTER(_C.c_int)
bind_conex_abi(_lib)
_lib.CONEXB200_CreateBatch.restype = _C.c_void_p
_lib.CONEXB200_NumberOfConstraints.argtypes = [_C.c_void_p]
_lib.CONEXB200_CreateBatch.argtypes = [_C.POINTER(_C.c_void_p), _C.c_int]
_lib.CONEXB200_DeleteBatch.argtypes = [_C.c_void_p]
_lib.CONEXB200_BatchMaximize.argtypes = [_C.c_void_p, _dp, _C.POINTER(CONEX_SolverConfiguration), _dp, _ip]
_lib.CONEXB200_BatchGetResults.argtypes = [_C.c_void_p, _ip, _dp, _dp, _dp]
_lib.CONEXB200_BatchUpdateConstraintData.argtypes = [_C.c_void_p, _C.c_int, _C.c_int, _C.c_int, _dp]
_lib.CONEXB200_BatchConstraintDataShape.argtypes = [_C.c_void_p, _C.c_int, _ip, _ip]


_lib.CONEXB200_SetKKTSolverKind.argtypes = [_C.c_void_p, _C.c_int]
_lib.CONEXB200_SetKKTSolverKind.restype = None
_lib.CONEXB200_GetNumberOfSupernodes.argtypes = [_C.c_void_p]
_lib.CONEXB200_SetCollective.argtypes = [_C.c_void_p, _C.c_int]
_lib.CONEXB200_SetCollective.restype = None


def device_available():
    return bool(_lib.CONEXB200_DeviceAvailable())


class Errors:
    """interfaces/python/ConexProgram.py `Errors`."""

    def __init__(self):
        self.Ax_minus_b = 0.0
        self.x_dot_s = 0.0
        self.min_eig_S = []
        self.min_eig_X = []


class Solution:
    def __init__(self):
        self.y = None
        self.status = 0


def _ptr(a):
    return a.ctypes.data_as(_dp)


class Conex:
    """Mirror of the reference's `Conex` class for the dense-LMI hot path."""

    def __init__(self, m=-1, library=None):
        # `library`: a ctypes library speaking the CONEX_* ABI (bind_conex_abi); default: the product
        self._lib = library if library is not None else _lib
        # extension entry point of whichever library is bound (the product, or the oracle in the CPU suite)
        self._count = getattr(self._lib, "CONEXB200_NumberOfConstraints", None) or self._lib.ORACLE_NumberOfConstraints
        self._count.argtypes = [_C.c_void_p]
        self.a = _C.c_void_p(self._lib.CONEX_CreateConeProgram())
        if not self.a:
            raise NameError("Failed to create program (is a B200 visible?).")
        if m >= 0:
            self._lib.CONEX_SetNumberOfVariables(self.a, m)
        self.num_constraints = 0
        self.A = []
        self.variables = []  # per constraint: the variables its operator acts on (None: built entry by entry)
        self.c = []
        self.m = m

    def __del__(self):
        if getattr(self, "a", None) and getattr(self, "_lib", None) is not None:
            self._lib.CONEX_DeleteConeProgram(self.a)

    def DefaultConfiguration(self):
        # interfaces/python/ConexProgram.py:115-126
        config = CONEX_SolverConfiguration()
        self._lib.CONEX_SetDefaultOptions(_C.byref(config))
        config.inv_sqrt_mu_max = 1000
        config.maximum_mu = 1e20
        config.max_iterations = 100
        config.final_centering_steps = 1
        config.prepare_dual_variables = 1
        config.infeasibility_threshold = 1e8
        config.divergence_upper_bound = 1
        return config

    def AddDenseLinearMatrixInequality(self, A, c):
        """A: array of shape (n, n, m) (A[:, :, i] is the i-th matrix), c: (n, n)."""
        A = _np.asarray(A, dtype=_np.float64)
        n, m = A.shape[1], A.shape[2]
        packed = _np.ascontiguousarray(_np.stack([_np.asfortranarray(A[:, :, i]).ravel(order="F")
                                                  for i in range(m)]))
        cf = _np.asfortranarray(_np.asarray(c, dtype=_np.float64))
        self.n, self.m = n, m
        self.A.append(A)
        self.c.append(cf)
        self.variables.append(_np.arange(m))
        self._lib.CONEX_AddDenseLMIConstraint(self.a, _ptr(packed), n, n, m, _ptr(cf), n, n)
        self.num_constraints += 1

    def AddLinearInequality(self, A, c):
        """c - A y >= 0 (interfaces/python/ConexProgram.py:98-105)."""
        Af = _np.asfortranarray(_np.asarray(A, dtype=_np.float64))
        cf = _np.ascontiguousarray(_np.asarray(c, dtype=_np.float64).ravel())
        self._lib.CONEX_AddDenseLinearConstraint(self.a, _ptr(Af), Af.shape[0], Af.shape[1], _ptr(cf), cf.shape[0])
        self.m, self.n = Af.shape[1], Af.shape[0]
        self.A.append(Af)
        self.c.append(cf.reshape(-1, 1))
        self.variables.append(_np.arange(Af.shape[1]))
        self.num_constraints += 1

    def AddLinearInequalities(self, A, lb, ub):
        """lb <= A y <= ub; rows with lb == ub become equality constraints (ConexProgram.py:107-114)."""
        Af = _np.asfortranarray(_np.asarray(A, dtype=_np.float64))
        lbf = _np.ascontiguousarray(_np.asarray(lb, dtype=_np.float64).ravel())
        ubf = _np.ascontiguousarray(_np.asarray(ub, dtype=_np.float64).ravel())
        before = self._count(self.a)
        self._lib.CONEX_AddLinearInequalities(self.a, _ptr(Af), Af.shape[0], Af.shape[1], _ptr(lbf), lbf.shape[0],
                                         _ptr(ubf), ubf.shape[0])
        # the call adds zero, one or two constraints (an LP cone with one row per finite bound, an equality
        # block for the rows with lb == ub): record each with the size the library reports for it
        for i in range(before, self._count(self.a)):
            self.A.append(None)
            self.c.append(_np.zeros((self._lib.CONEX_GetDualVariableSize(self.a, i), 1)))
            self.variables.append(None)
            self.num_constraints += 1

    def _new(self, fn, *args):
        cid = _C.c_int(-1)
        if fn(self.a, *args, _C.byref(cid)) != 0:
            raise NameError("Failed to add constraint.")
        self.num_constraints += 1
        return cid.value

    def NewLinearMatrixInequality(self, order, hyper_complex_dim):
        cid = self._new(self._lib.CONEX_NewLinearMatrixInequality, order, hyper_complex_dim)
        self.c.append(_np.zeros((order, order)))
        self.A.append(None)
        self.variables.append(None)
        return cid

    def NewLorentzConeConstraint(self, order):
        cid = self._new(self._lib.CONEX_NewLorentzConeConstraint, order)
        self.c.append(_np.zeros((order + 1, 1)))
        self.A.append(None)
        self.variables.append(None)
        return cid

    def NewLinearInequality(self, num_rows):
        cid = self._new(self._lib.CONEX_NewLinearInequality, num_rows)
        self.c.append(_np.zeros((num_rows, 1)))
        self.A.append(None)
        self.variables.append(None)
        return cid

    def UpdateLinearOperator(self, constraint, value, variable, row, col=0, hyper_complex_dim=0):
        if self._lib.CONEX_UpdateLinearOperator(self.a, constraint, float(value), variable, row, col,
                                           hyper_complex_dim) != 0:
            raise NameError("Failed to update operator.")

    def UpdateAffineTerm(self, constraint, value, row, col=0, hyper_complex_dim=0):
        if self._lib.CONEX_UpdateAffineTerm(self.a, constraint, float(value), row, col, hyper_complex_dim) != 0:
            raise NameError("Failed to update affine term.")

    def AddSparseLinearMatrixInequality(self, A, c, variables):
        A = _np.asarray(A, dtype=_np.float64)
        n, k = A.shape[1], A.shape[2]
        if max(variables) + 1 > self.m:
            raise NameError("Invalid sparse LMI.")
        packed = _np.ascontiguousarray(_np.stack([_np.asfortranarray(A[:, :, i]).ravel(order="F")
                                                  for i in range(k)]))
        cf = _np.asfortranarray(_np.asarray(c, dtype=_np.float64))
        v = (_C.c_long * k)(*[int(x) for x in variables])
        self.A.append(A)
        self.c.append(cf)
        self.variables.append(_np.array([int(x) for x in variables]))
        self._lib.CONEX_AddSparseLMIConstraint(self.a, _ptr(packed), n, n, k, _ptr(cf), n, n, v, k)
        self.num_constraints += 1

    # ---- conex-b200 extensions (include/conex_b200.h) ----
    def SetKKTSolverKind(self, kind):
        """0: chosen from the cones' variable sets (default), 1: one dense supernode, 2: multifrontal
        (cones on overlapping variable subsets, AddSparseLinearMatrixInequality). Before the first solve."""
        _lib.CONEXB200_SetKKTSolverKind(self.a, int(kind))

    def NumberOfSupernodes(self):
        """Supernodes of the KKT solver in use (1 = dense); valid after the first solve."""
        return _lib.CONEXB200_GetNumberOfSupernodes(self.a)

    def SetCollective(self, collective=True):
        """Every rank of the process-wide communicator builds this same program and solves in lock step
        (the Cholesky of large Schur complements is then factored across the GPUs)."""
        _lib.CONEXB200_SetCollective(self.a, int(bool(collective)))

    def Maximize(self, b, config=None):
        if config is None:
            config = self.DefaultConfiguration()
        b = _np.ascontiguousarray(_np.asarray(b, dtype=_np.float64).ravel())
        if b.shape[0] != self.m:
            raise NameError("Cost vector dimension does not match number of variables.")
        sol = Solution()
        sol.y = _np.ones(self.m)
        sol.status = self._lib.CONEX_Maximize(self.a, _ptr(b), self.m, _C.byref(config), _ptr(sol.y), self.m)
        return sol

    def GetDualVariables(self):
        x = []
        for i in range(self.num_constraints):
            r, c = self.c[i].shape[0], self.c[i].shape[1]
            size = self._lib.CONEX_GetDualVariableSize(self.a, i)
            if r * c != size:
                r, c = size, 1
            xi = _np.zeros(r * c)
            self._lib.CONEX_GetDualVariable(self.a, i, _ptr(xi), r, c)
            x.append(xi.reshape((r, c), order="F"))
        return x

    def ComputeErrors(self, y, xa, b):
        """interfaces/python/ConexProgram.py:243-277: slacks c_i - A_i y of every constraint and the
        residuals |b - sum_i A_i' x_i|, sum_i <x_i, s_i>, smallest eigenvalues of s_i and x_i."""
        y = _np.asarray(y, dtype=_np.float64).ravel()
        b = _np.asarray(b, dtype=_np.float64).ravel()
        err = Errors()
        slacks = []
        Ax = _np.zeros(self.m)
        for i in range(self.num_constraints):
            if self.A[i] is None:
                raise NameError("ComputeErrors needs the operator: constraint %d was built entry by entry." % i)
            A, c = self.A[i], _np.asarray(self.c[i], dtype=_np.float64)
            variables = self.variables[i]
            x = _np.asarray(xa[i], dtype=_np.float64)
            if A.ndim == 3:   # LMI: A[:, :, k] is the matrix of variable variables[k]
                s = c - _np.tensordot(A, y[variables], axes=([2], [0]))
                Ax[variables] += _np.tensordot(A, x, axes=([0, 1], [0, 1]))
                err.x_dot_s += float(_np.trace(s @ x))
                err.min_eig_S.append(float(_np.linalg.eigvalsh(0.5 * (s + s.T)).min()))
                err.min_eig_X.append(float(_np.linalg.eigvalsh(0.5 * (x + x.T)).min()))
            else:             # linear inequality: rows x variables
                s = c.ravel() - A @ y[variables]
                Ax[variables] += A.T @ x.ravel()
                err.x_dot_s += float(s @ x.ravel())
                err.min_eig_S.append(float(s.min()))
                err.min_eig_X.append(float(x.min()))
            slacks.append(s)
        err.Ax_minus_b = float(_np.linalg.norm(b - Ax))
        return slacks, err

    def GetIterationNumberStats(self, num):
        stats = CONEX_IterationStats()
        self._lib.CONEX_GetIterationStats(self.a, _C.byref(stats), num)
        return stats

    def GetIterationStats(self):
        last = self.GetIterationNumberStats(-1).iteration_number
        return [self.GetIterationNumberStats(i) for i in range(last + 1)]


class ConexBatch:
    """Many structurally identical `Conex` programs solved in lock step on one GPU
    (CONEXB200_CreateBatch / CONEXB200_BatchMaximize, include/conex_b200.h). No counterpart in the
    reference, which solves such programs one after the other.

    The programs may combine LP, second-order and dense LMI cones with equality constraints (e.g. the
    lb == ub rows of AddLinearInequalities). Each cone or equality block acts on all variables or on a
    list of distinct variables (a dense LMI added with a variable list, the LP and second-order cones of
    CONEXB200_AddSparseLinearConstraint / CONEXB200_AddSparseSocConstraint); every program must have
    the same constraints, on the same variable lists, in the same order. With equality constraints the
    KKT systems are factored by a batched regularised LDL^T, and iterative refinement, or a line
    search on programs of LP cones and equalities only, is refused.

    A batch lives across solves: `config.initialization_mode = 1` warm-starts every program from the
    iterate of the previous Maximize (an error before the first one), and UpdateConstraintData
    changes the programs' data in place between solves."""

    def __init__(self, programs):
        self.count = len(programs)
        self.m = programs[0].m
        handles = (_C.c_void_p * self.count)(*[p.a for p in programs])
        self.h = _C.c_void_p(_lib.CONEXB200_CreateBatch(handles, self.count))
        if not self.h:
            raise NameError("Failed to create the batch (programs must have identical structure).")

    def __del__(self):
        if getattr(self, "h", None):
            _lib.CONEXB200_DeleteBatch(self.h)

    def Maximize(self, b, config=None):
        """b: (count, m). Returns a list of Solution."""
        if config is None:
            config = programs_default_configuration()
        b = _np.ascontiguousarray(_np.asarray(b, dtype=_np.float64))
        if b.shape != (self.count, self.m):
            raise NameError("Cost matrix dimension does not match the batch.")
        y = _np.zeros((self.count, self.m))
        status = (_C.c_int * self.count)()
        if _lib.CONEXB200_BatchMaximize(self.h, _ptr(b), _C.byref(config), _ptr(y), status) < 0:
            raise NameError("Batched solve failed.")
        out = []
        for p in range(self.count):
            s = Solution()
            s.y, s.status = y[p], status[p]
            out.append(s)
        return out

    def UpdateConstraintData(self, constraint, first, data):
        """Replaces columns [first, first + ncols) of the data of constraint `constraint` (numbered like
        GetDualVariables) in every program; data has shape (count, rows, ncols), data[p] for program p.
        Cones: column j < m holds the coefficients of y_j (LP / second-order: column j of A; LMI: the
        column-major vec of A_j, rows = n * n), column m the affine term; a cone on a list of m_k
        variables v has m_k + 1 columns, column j < m_k for y[v_j] and column m_k the affine term.
        Equality constraints: column j < nvars is column j of A, column nvars is b."""
        data = _np.asarray(data, dtype=_np.float64)
        rows, columns = _C.c_int(), _C.c_int()
        if _lib.CONEXB200_BatchConstraintDataShape(self.h, int(constraint), _C.byref(rows), _C.byref(columns)) != 0:
            raise NameError("The batch has no constraint %d." % constraint)
        if data.ndim != 3 or data.shape[0] != self.count or data.shape[1] != rows.value:
            raise NameError("Constraint data must have shape (%d, %d, columns)." % (self.count, rows.value))
        blocks = _np.ascontiguousarray(data.transpose(0, 2, 1))
        if _lib.CONEXB200_BatchUpdateConstraintData(self.h, int(constraint), int(first), data.shape[2],
                                                    _ptr(blocks)) != 0:
            raise NameError("Failed to update the constraint data (constraint or column range out of range).")


def programs_default_configuration():
    config = CONEX_SolverConfiguration()
    _lib.CONEX_SetDefaultOptions(_C.byref(config))
    return config
