"""K2 of the symmetric Schur assembly emulated on the 8-bit integer tensor cores (device/ozaki.cu).

1. The int8 slices and column exponents are those of a numpy restatement of the slicing, and the Gram is bit-identical
   to the same arithmetic done exactly on those slices (level sums per 2^15 K chunk as exact integers, converted and
   added in the kernel's order), at ragged shapes, K not a multiple of the chunk or of the 32-byte k-step, columns with
   a 2^60 spread of magnitudes, all-zero columns and denormal-range columns.
2. Against the DMMA Gram on the packed scaled matrices X = L^T A_i L of a MaxCut instance (n = 400, the C2 family), at
   W = I (the cold start) and at a W with the eigenvalue spread of a late interior-point iterate: every entry within
   the documented bound K 2^-50.8 max|X_i| max|X_j| plus the FP64 product's own rounding.
3. Two runs are bit-identical."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SLICES = 8
CHUNK = 1 << 15


@pytest.fixture(scope="module")
def lib():
    import devlib
    L = devlib.product().lib
    vp = C.c_void_p
    L.cxb_gram_emulated_workspace.restype = C.c_size_t
    L.cxb_gram_emulated_workspace.argtypes = [C.c_int, C.c_long]
    L.cxb_gram_slices.argtypes = [vp, C.c_int, C.c_long, vp, C.c_long, vp]
    L.cxb_gram_emulated.argtypes = [vp, C.c_int, C.c_int, C.c_long, vp, C.c_long, vp, C.c_long, vp]
    L.cxb_packed_symmetric_size.restype = C.c_size_t
    L.cxb_packed_symmetric_size.argtypes = [C.c_int]
    L.cxb_schur_dense_lmi_sym_scale.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp, C.c_int, vp, vp]
    L.cxb_dgemm.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, vp, C.c_long, C.c_long, vp,
                            C.c_long, C.c_long, C.c_double, vp, C.c_long, C.c_long, C.c_int, C.c_int]
    return L


def numpy_slices(X):
    """X: K x M. Returns digits (SLICES x M x K, int8) and exponents e_j with max|X[:, j]| < 2^e_j."""
    K, M = X.shape
    mx = np.abs(X).max(axis=0)
    e = np.where(mx > 0, np.frexp(mx)[1], 0).astype(np.int32)
    r = np.ldexp(X, (6 - e)[None, :])
    D = np.empty((SLICES, M, K), dtype=np.int8)
    for t in range(SLICES):
        d = np.rint(r)
        D[t] = d.T.astype(np.int8)
        r = (r - d) * 128.0
    return D, e


def exact_gram(D, e, N):
    """The kernel's arithmetic on the slices: exact integer level sums per K chunk (float64 products of digits and
    their sums stay below 2^53), added into FP64 chunk by chunk and level by level, then scaled by 2^(e_i + e_j - 12)."""
    _, M, K = D.shape
    acc = np.zeros((M, N))
    F = D.astype(np.float64)
    for k0 in range(0, K, CHUNK):
        Fc = F[:, :, k0:k0 + CHUNK]
        for lv in range(SLICES):
            s = np.zeros((M, N))
            for t in range(lv + 1):
                s += Fc[t] @ Fc[lv - t, :N].T
            acc += np.ldexp(1.0, -7 * lv) * s
    return np.ldexp(acc, (e[:, None] + e[None, :N] - 12).astype(np.int32))


def run_emulated(L, X, N):
    import torch
    import devlib
    K, M = X.shape
    dX = torch.from_numpy(np.asfortranarray(X).ravel(order="F")).cuda()
    work = torch.zeros(L.cxb_gram_emulated_workspace(M, K), dtype=torch.uint8, device="cuda")
    dH = torch.full((M * N,), float("nan"), dtype=torch.float64, device="cuda")
    assert L.cxb_gram_emulated(None, M, N, K, devlib.ptr(dX), K, devlib.ptr(dH), M, devlib.ptr(work)) == 0
    torch.cuda.synchronize()
    H = dH.cpu().numpy().reshape(N, M).T
    D, e = untile(work.cpu().numpy(), M, K)
    return H, D, e


def untile(w, M, K):
    """The workspace's digits as D[t][j][k] and its exponents. Layout (ozaki.cu): 128-row blocks, then 32-byte k-steps,
    then slices, each 128 rows x 32 bytes with the 16-byte half h of row r at h ^ ((r >> 2) & 1); zero padding."""
    nb, ksteps = (M + 127) // 128, (K + 31) // 32
    size = nb * ksteps * SLICES * 128 * 32
    arr = w[:size].view(np.int8).reshape(nb, ksteps, SLICES, 128, 2, 16)
    sw = (np.arange(128) >> 2) & 1
    phys = np.stack([sw, 1 - sw], axis=1)  # physical half of logical half 0, 1
    logical = np.take_along_axis(arr, phys[None, None, None, :, :, None], axis=4)
    full = logical.reshape(nb, ksteps, SLICES, 128, 32).transpose(2, 0, 3, 1, 4).reshape(SLICES, nb * 128, ksteps * 32)
    assert not full[:, M:, :].any() and not full[:, :, K:].any()
    e = w[size:size + 4 * M].view(np.int32).copy()
    return full[:, :M, :K], e


def awkward_operand(rng, K, M):
    X = rng.standard_normal((K, M))
    X[:, 1] *= 2.0 ** 60                              # 2^60 spread of column magnitudes
    X[:, 2] *= 2.0 ** -60
    X[:, 3] = 0.0                                     # all-zero column
    X[:, 4] = rng.standard_normal(K) * 1e-310         # denormal range
    X[:, 5] = rng.standard_normal(K) * 2.0 ** rng.integers(-60, 60, K)  # 2^120 spread inside one column
    X[::7, 6] = 0.0
    return X


@pytest.mark.parametrize("K,M,N", [(4096, 130, 129), (CHUNK + 48, 300, 299), (2 * CHUNK + 4096, 257, 257)])
def test_emulated_gram_matches_exact_slice_arithmetic(lib, K, M, N):
    rng = np.random.default_rng(K + M)
    X = awkward_operand(rng, K, M)
    H, D, e = run_emulated(lib, X, N)
    Dref, eref = numpy_slices(X)
    assert np.array_equal(e, eref)
    assert np.array_equal(D, Dref)
    ref = exact_gram(D, e, N)
    low = np.tril(np.ones((M, N), dtype=bool))
    assert np.array_equal(H[low], ref[low])


def maxcut_scaled(L, n, W):
    """Packed X = [L^T A_i L, L^T C L, I] of a MaxCut instance from K1 (cxb_schur_dense_lmi_sym_scale)."""
    import torch
    import devlib
    from conex_b200.workloads import maxcut_lmi
    mats, Cm, _ = maxcut_lmi(n, 11)
    m = len(mats)
    dA = torch.from_numpy(np.concatenate([np.asfortranarray(A).ravel(order="F") for A in mats + [Cm]])).cuda()
    kp = L.cxb_packed_symmetric_size(n)
    dX = devlib.dzeros((m + 2) * kp)
    dT = devlib.dzeros(n * n * 8)
    dL = devlib.dzeros(n * n)
    info = devlib.izeros(2)
    assert L.cxb_schur_dense_lmi_sym_scale(None, n, m, devlib.ptr(dA), devlib.ptr(devlib.to_dev(W)), devlib.ptr(dX),
                                           devlib.ptr(dT), 8, devlib.ptr(dL), devlib.ptr(info)) == 0
    assert int(info.cpu()[0]) == 0
    return dX, m, kp


@pytest.mark.parametrize("iterate", ["cold_start", "late"])
def test_emulated_gram_within_bound_of_dmma_gram(lib, iterate):
    import torch
    import devlib
    n = 400
    rng = np.random.default_rng(5)
    if iterate == "cold_start":
        W = np.eye(n)
    else:
        Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
        W = (Q * np.logspace(-8, 0, n)) @ Q.T
        W = 0.5 * (W + W.T)
    dX, m, kp = maxcut_scaled(lib, n, W)
    M, N = m + 2, m + 1
    work = torch.zeros(lib.cxb_gram_emulated_workspace(M, kp), dtype=torch.uint8, device="cuda")
    dH = devlib.dzeros(M * N)
    dR = devlib.dzeros(M * N)
    assert lib.cxb_gram_emulated(None, M, N, kp, devlib.ptr(dX), kp, devlib.ptr(dH), M, devlib.ptr(work)) == 0
    assert lib.cxb_dgemm(None, 1, 0, M, N, kp, 1.0, devlib.ptr(dX), kp, 0, devlib.ptr(dX), kp, 0, 0.0,
                         devlib.ptr(dR), M, 0, 1, 1) == 0
    torch.cuda.synchronize()
    H = dH.cpu().numpy().reshape(N, M).T
    R = dR.cpu().numpy().reshape(N, M).T
    X = dX.cpu().numpy().reshape(M, kp)
    mx = np.abs(X).max(axis=1)
    absX = np.abs(X)
    u = 2.0 ** -53
    bound = kp * 2.0 ** -50.8 * np.outer(mx, mx[:N]) + 2 * kp * u * (absX @ absX[:N].T)
    low = np.tril(np.ones((M, N), dtype=bool))
    err = np.abs(H - R)
    assert (err[low] <= bound[low]).all(), float((err[low] / bound[low]).max())


def test_emulated_gram_is_bit_identical_across_runs(lib):
    rng = np.random.default_rng(3)
    X = awkward_operand(rng, CHUNK + 4096, 260)
    H1, _, _ = run_emulated(lib, X, 259)
    H2, _, _ = run_emulated(lib, X, 259)
    low = np.tril(np.ones(H1.shape, dtype=bool))
    assert np.array_equal(H1[low], H2[low])
