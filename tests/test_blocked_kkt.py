"""The blocked factorisations of KKT systems larger than shared memory (BlockedPotrf / BlockedLdlt of
small_cone_math.cuh, behind cxb_small_potrf / cxb_small_ldlt above N = 170 / 169) on the host stand-in of the CTA
(tests/emul/emul_blocked_kkt.cc): block columns of 32, so the sizes below cover one partial block, exact blocks, a
ragged last block and several trailing updates. Compared with numpy restatements of the contract: the Cholesky factor
and its failing column, the pivot order of Eigen::RLDLT, the signed factor and its regularisation flag.
"""
import numpy as np
import pytest

from kkt_backend import KktBackend
from test_small_ldlt import kkt_matrix, regularised_ldlt, rldlt_pivot_order, tricky_diagonals

NB = 32
SIZES = [1, 2, NB - 1, NB, NB + 1, 2 * NB + 3, 171, 300]


@pytest.fixture(scope="module")
def be():
    return KktBackend("emul")


def spd(rng, N):
    R = rng.uniform(-1, 1, size=(N, N + 2))
    return R @ R.T / N + np.eye(N)


def rel(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


@pytest.mark.parametrize("N", SIZES)
def test_cholesky_matches_numpy(be, N):
    rng = np.random.Generator(np.random.PCG64(11 + N))
    H = np.stack([spd(rng, N) for _ in range(3)])
    out, info, _ = be.potrf(H)
    assert info.tolist() == [0, 0, 0]
    for p in range(3):
        assert rel(np.tril(out[p]), np.linalg.cholesky(H[p])) < 1e-12, p


@pytest.mark.parametrize("N", [2 * NB + 3, 171])
def test_cholesky_reports_first_failing_column(be, N):
    """The leading minor stops being positive at column f of the second block (a negative pivot, a zero pivot, a NaN
    pivot); the programs around it factor normally."""
    rng = np.random.Generator(np.random.PCG64(3 * N))
    cols = [NB + 5, NB + NB - 1, NB]
    H = [spd(rng, N)]
    for f, new_pivot in zip(cols, [-1.0, 0.0, np.nan]):
        M = spd(rng, N)
        schur = M[f, f] - M[f, :f] @ np.linalg.solve(M[:f, :f], M[:f, f])
        M[f, f] += new_pivot - schur if np.isfinite(new_pivot) else np.nan
        if new_pivot == 0.0:
            M[f, f] -= 1e-3  # rounding can leave +-tiny instead of 0; make it clearly not > 0
        H.append(M)
    H.append(spd(rng, N))
    _, info, _ = be.potrf(np.stack(H))
    assert info.tolist() == [0] + [f + 1 for f in cols] + [0]


@pytest.mark.parametrize("N", SIZES)
def test_ldlt_matches_restatement(be, N):
    rng = np.random.Generator(np.random.PCG64(5 + N))
    rows = N // 4
    K = np.stack([kkt_matrix(rng, N - rows, rows) for _ in range(3)])
    L, perm, signs, info, _, Kafter = be.ldlt(K)
    assert np.array_equal(Kafter, K)
    for p in range(3):
        order = rldlt_pivot_order(np.diag(K[p]))
        assert perm[p].tolist() == order
        Lr, sr, reg = regularised_ldlt(K[p][np.ix_(order, order)])
        assert np.array_equal(signs[p], sr)
        assert info[p] == reg
        assert rel(np.tril(L[p]), Lr) < 1e-12, p


@pytest.mark.parametrize("N", [NB + 1, 171])
def test_ldlt_tricky_diagonals(be, N):
    """Ties, exact zeros and +-d of equal magnitude: same pivot order, signs and regularisation flag as the
    restatement."""
    rng = np.random.Generator(np.random.PCG64(100 + N))
    K = []
    for d in tricky_diagonals(N, rng):
        R = 1e-3 * rng.uniform(-1, 1, size=(N, N))
        M = 0.5 * (R + R.T)
        np.fill_diagonal(M, d)
        K.append(M)
    K = np.stack(K)
    L, perm, signs, info, _, _ = be.ldlt(K)
    for p in range(len(K)):
        order = rldlt_pivot_order(np.diag(K[p]))
        assert perm[p].tolist() == order
        Lr, sr, reg = regularised_ldlt(K[p][np.ix_(order, order)])
        assert info[p] == reg, p
        assert np.array_equal(signs[p], sr), p
    assert info.tolist()[2] == 1  # the all-zero diagonal


def test_masked_programs_are_untouched(be):
    rng = np.random.Generator(np.random.PCG64(9))
    B, N = 4, 2 * NB + 3
    active = np.array([1, 0, 1, 0], dtype=np.int32)
    sentinel = rng.uniform(-1, 1, size=(B, N, N))
    H = np.stack([spd(rng, N) for _ in range(B)])
    out, info, _ = be.potrf(H, active=active, H_init=sentinel)
    K = np.stack([kkt_matrix(rng, N - 7, 7) for _ in range(B)])
    L, perm, signs, linfo, _, _ = be.ldlt(K, active=active, L_init=sentinel)
    for p in range(B):
        if active[p]:
            assert info[p] == 0 and linfo[p] == 0
        else:
            assert np.array_equal(out[p], sentinel[p]) and info[p] == -3
            assert np.array_equal(L[p], sentinel[p]) and linfo[p] == -3
            assert (perm[p] == -7).all() and (signs[p] == 5.0).all()
