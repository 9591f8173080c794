"""The batched regularised LDL^T of small KKT systems with equality multipliers (cxb_small_ldlt /
cxb_small_ldlt_solve, small_cone_math.cuh SmallLdlt / SmallLdltSolve): the pivot order of Eigen::RLDLT from the
diagonal, the signed factorisation L S L^T of P K P^T with its regularisation of tiny pivots, and the solve.

The same checks run on the CPU through the host stand-in of the CTA (tests/emul/emul_ldlt.cc) and, marked gpu, through the real
kernels; on the GPU the factors are also compared with the single-matrix path (cxb_sym_permute_lower +
cxb_ldlt_lower) that CONEX_Maximize uses for programs with equality constraints.
"""
import ctypes as C

import numpy as np
import pytest

from harness import dptr
from ldlt_backend import LdltBackend


@pytest.fixture(scope="module", params=["emul", pytest.param("device", marks=pytest.mark.gpu)])
def be(request):
    return LdltBackend(request.param)


def rldlt_pivot_order(diag):
    """Restatement of RldltPivotOrder (host/cone_program.cc): at step k the first largest |d| among positions k..
    of the current arrangement is swapped to position k."""
    d = np.abs(np.asarray(diag, dtype=np.float64)).tolist()
    at = list(range(len(d)))
    for k in range(len(d)):
        p = k + int(np.argmax(d[k:]))
        d[k], d[p] = d[p], d[k]
        at[k], at[p] = at[p], at[k]
    return at


def regularised_ldlt(M):
    """L S L^T of M without pivoting, the rule of LdltDiagKernel (cholesky.cu): |d| <= 1e-9 becomes -1e-9 when
    d < 0, +1e-9 otherwise."""
    A = np.array(M, dtype=np.float64)
    N = A.shape[0]
    L = np.zeros((N, N))
    s = np.zeros(N)
    reg = 0
    for j in range(N):
        d = A[j, j]
        if not abs(d) > 1e-9:
            d = -1e-9 if d < 0 else 1e-9
            reg = 1
        s[j] = -1.0 if d < 0 else 1.0
        col = A[j + 1:, j] / np.sqrt(abs(d))
        L[j, j] = np.sqrt(abs(d))
        L[j + 1:, j] = s[j] * col
        A[j + 1:, j + 1:] -= s[j] * np.outer(col, col)
    return L, s, reg


def kkt_matrix(rng, m, rows):
    R = rng.uniform(-1, 1, size=(m, m + 2))
    N = m + rows
    K = np.zeros((N, N))
    K[:m, :m] = R @ R.T + 0.5 * np.eye(m)
    if rows:
        A = rng.uniform(-1, 1, size=(rows, m))
        K[m:, :m] = A
        K[:m, m:] = A.T
    return K


def product_pivot_order(diag):
    import devlib
    L = devlib.product().lib
    L.CONEXB200_RldltPivotOrder.argtypes = [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int)]
    d = np.ascontiguousarray(np.asarray(diag, dtype=np.float64))
    perm = (C.c_int * len(d))()
    L.CONEXB200_RldltPivotOrder(len(d), dptr(d), perm)
    return list(perm)


def tricky_diagonals(N, rng):
    """Diagonals with exact ties, +-d of equal magnitude, exact zeros and all-equal entries."""
    out = []
    d = rng.choice([-3.0, -1.0, 0.0, 1.0, 2.0, 3.0], size=N)
    out.append(d)
    out.append(np.full(N, 1.5))
    out.append(np.zeros(N))
    e = rng.uniform(0.5, 4.0, size=N)
    e[N // 2:] = 0.0  # a multiplier block
    if N > 3:
        e[1] = -e[0]
        e[3] = e[2]
    out.append(e)
    out.append(np.where(np.arange(N) % 2 == 0, 2.0, -2.0))
    return out


@pytest.mark.parametrize("N", [1, 2, 17, 48, 100])
def test_pivot_order(be, N):
    rng = np.random.Generator(np.random.PCG64(100 + N))
    diags = tricky_diagonals(N, rng)
    K = []
    for d in diags:
        R = 1e-3 * rng.uniform(-1, 1, size=(N, N))
        M = 0.5 * (R + R.T)
        np.fill_diagonal(M, d)
        K.append(M)
    _, perm, _, _, _, _ = be.ldlt(np.stack(K))
    for p, d in enumerate(diags):
        ref = rldlt_pivot_order(d)
        assert perm[p].tolist() == ref, (p, d)
        if be.kind == "device":
            assert product_pivot_order(d) == ref


@pytest.mark.parametrize("m,rows", [(1, 0), (1, 1), (12, 5), (40, 8), (80, 20)])
def test_kkt_factor_and_solve(be, m, rows):
    rng = np.random.Generator(np.random.PCG64(7 * m + rows))
    B = 6
    N = m + rows
    K = np.stack([kkt_matrix(rng, m, rows) for _ in range(B)])
    L, perm, signs, info, handles, Kafter = be.ldlt(K)
    assert (info == 0).all()
    assert np.array_equal(Kafter, K)  # K is not modified
    for p in range(B):
        assert perm[p].tolist() == rldlt_pivot_order(np.diag(K[p]))
        P = K[p][np.ix_(perm[p], perm[p])]
        Lp = np.tril(L[p])
        assert set(signs[p].tolist()) <= {-1.0, 1.0}
        assert int((signs[p] < 0).sum()) == rows  # the inertia of a KKT matrix with full-rank A
        err = np.abs(Lp @ np.diag(signs[p]) @ Lp.T - P).max() / np.abs(K[p]).max()
        assert err < 1e-12, (p, err)
    X = rng.uniform(-1, 1, size=(B, N))
    sol = be.ldlt_solve(handles, B, N, X)
    for p in range(B):
        ref = np.linalg.solve(K[p], X[p])
        assert np.abs(sol[p] - ref).max() <= 1e-9 * max(1.0, np.abs(ref).max()), p


def test_zero_pivots_are_regularised(be):
    # [[0, 1], [1, 0]] blocks: every diagonal entry is 0, the order stays the identity, the first pivot of each
    # block becomes +1e-9 and the second -1e9 (RLDLT.h:378-389)
    J = np.array([[0.0, 1.0], [1.0, 0.0]])
    K0 = np.kron(np.eye(3), J)
    K1 = np.zeros((6, 6))
    K1[:2, :2] = J
    K1[2:, 2:] = np.diag([2.0, 3.0, -1.0, 5.0])
    K2 = np.diag([4.0, 3.0, 2.0, 1.0, 1.5, 2.5])
    K = np.stack([K0, K1, K2])
    L, perm, signs, info, _, _ = be.ldlt(K)
    assert info.tolist() == [1, 1, 0]
    for p in range(3):
        order = rldlt_pivot_order(np.diag(K[p]))
        assert perm[p].tolist() == order
        Lr, sr, reg = regularised_ldlt(K[p][np.ix_(order, order)])
        assert reg == info[p]
        assert np.array_equal(signs[p], sr)
        assert np.abs(np.tril(L[p]) - Lr).max() <= 1e-12 * np.abs(Lr).max()
    assert signs[0].tolist() == [1.0, -1.0] * 3


def test_inactive_programs_are_untouched(be):
    rng = np.random.Generator(np.random.PCG64(5))
    B, m, rows = 5, 9, 3
    N = m + rows
    K = np.stack([kkt_matrix(rng, m, rows) for _ in range(B)])
    active = np.array([1, 0, 1, 0, 1], dtype=np.int32)
    L0 = rng.uniform(-1, 1, size=(B, N, N))
    L, perm, signs, info, handles, Kafter = be.ldlt(K, active=active, L_init=L0)
    assert np.array_equal(Kafter, K)
    for p in range(B):
        if active[p]:
            assert info[p] == 0 and perm[p].tolist() == rldlt_pivot_order(np.diag(K[p]))
        else:
            assert info[p] == -3 and (perm[p] == -7).all() and (signs[p] == 5.0).all()
            assert np.array_equal(L[p], L0[p])
    X = rng.uniform(-1, 1, size=(B, N))
    sol = be.ldlt_solve(handles, B, N, X, active=active)
    for p in range(B):
        if active[p]:
            assert np.abs(sol[p] - np.linalg.solve(K[p], X[p])).max() <= 1e-9 * max(1.0, np.abs(sol[p]).max())
        else:
            assert np.array_equal(sol[p], X[p])


@pytest.mark.gpu
@pytest.mark.parametrize("m,rows", [(12, 5), (40, 8), (80, 20)])
def test_device_batch_matches_single_matrix_ldlt(m, rows):
    """The batched factor equals cxb_sym_permute_lower + cxb_ldlt_lower on the same matrix (L and S)."""
    import devlib as dev
    import torch
    be = LdltBackend("device")
    lib = dev.product().lib
    vp = C.c_void_p
    lib.cxb_ldlt_worksize.restype = C.c_size_t
    lib.cxb_ldlt_worksize.argtypes = [C.c_int]
    lib.cxb_sym_permute_lower.argtypes = [vp, C.c_int, vp, C.c_long, vp, vp, C.c_long]
    lib.cxb_ldlt_lower.argtypes = [vp, C.c_int, vp, C.c_long, vp, vp, vp]
    rng = np.random.Generator(np.random.PCG64(m * rows))
    N = m + rows
    B = 4
    K = np.stack([kkt_matrix(rng, m, rows) for _ in range(B)])
    # a tiny pivot in one program, so the regularisation is compared too
    K[1][m - 1, :] = 0.0
    K[1][:, m - 1] = 0.0
    L, perm, signs, info, _, _ = be.ldlt(K)
    for p in range(B):
        order = product_pivot_order(np.diag(K[p]))
        assert perm[p].tolist() == order
        dK = dev.to_dev(np.tril(K[p]))
        dperm = torch.from_numpy(np.array(order, dtype=np.int32)).cuda()
        dKp = dev.dzeros(N * N)
        assert lib.cxb_sym_permute_lower(None, N, dev.ptr(dK), N, dev.ptr(dperm), dev.ptr(dKp), N) == 0
        ds = dev.dzeros(N)
        work = dev.dzeros(lib.cxb_ldlt_worksize(N))
        dinfo = dev.izeros(2)
        assert lib.cxb_ldlt_lower(None, N, dev.ptr(dKp), N, dev.ptr(ds), dev.ptr(work), dev.ptr(dinfo)) == 0
        Lref = np.tril(dev.from_dev(dKp, N, N))
        assert np.array_equal(signs[p], dev.from_dev(ds))
        assert int(info[p]) == dinfo.cpu().tolist()[1]
        assert np.abs(np.tril(L[p]) - Lref).max() <= 1e-12 * np.abs(Lref).max(), p
