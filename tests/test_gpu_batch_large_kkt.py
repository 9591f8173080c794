"""Batched solves whose KKT systems do not fit in shared memory: cxb_small_potrf above N = 170 and cxb_small_ldlt above
N = 169 use the blocked kernels (cxb_small_potrf_blocked / cxb_small_ldlt_blocked, block columns of 32, DMMA trailing
updates). Kernel level: against numpy restatements of the contract, against the single-matrix device path that
CONEX_Maximize uses, and against the shared-memory kernels where those run (1e-12: the summation order differs); masked
programs and K are left bit for bit as they were. Whole solves: long MPC horizons (conex_b200.workloads.mpc_problem)
against the CPU oracle on the zero-padded programs and CONEX_Maximize on the device, with the tolerances of
test_gpu_batch_subsets.py.
"""
import ctypes as C

import numpy as np
import pytest

from harness import add_cones, mpc_problem
from kkt_backend import KktBackend
from test_gpu_batch_subsets import (assert_parity, batch_outcome, check_both_references, make_batch, make_program,
                                    updated)
from test_small_ldlt import kkt_matrix, product_pivot_order, regularised_ldlt, rldlt_pivot_order

pytestmark = pytest.mark.gpu
NB = 32
vp = C.c_void_p


@pytest.fixture(scope="module")
def be():
    return KktBackend("device")


@pytest.fixture(scope="module")
def libs():
    import devlib
    from harness import oracle
    return oracle(), devlib.product()


def spd(rng, N):
    R = rng.uniform(-1, 1, size=(N, N + 2))
    return R @ R.T / N + np.eye(N)


def rel(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


def single_matrix_cholesky(H):
    import devlib as dev
    import torch
    lib = dev.product().lib
    lib.cxb_potrf_lower.argtypes = [vp, C.c_int, vp, C.c_long, vp, vp]
    N = H.shape[0]
    dH = dev.to_dev(np.tril(H))
    info = dev.izeros(1)
    assert lib.cxb_potrf_lower(None, N, dev.ptr(dH), N, None, dev.ptr(info)) == 0
    torch.cuda.synchronize()
    assert int(info.cpu()[0]) == 0
    return np.tril(dev.from_dev(dH, N, N))


def single_matrix_ldlt(K, order):
    import devlib as dev
    import torch
    lib = dev.product().lib
    lib.cxb_ldlt_worksize.restype = C.c_size_t
    lib.cxb_ldlt_worksize.argtypes = [C.c_int]
    lib.cxb_sym_permute_lower.argtypes = [vp, C.c_int, vp, C.c_long, vp, vp, C.c_long]
    lib.cxb_ldlt_lower.argtypes = [vp, C.c_int, vp, C.c_long, vp, vp, vp]
    N = K.shape[0]
    dK = dev.to_dev(np.tril(K))
    dperm = torch.from_numpy(np.array(order, dtype=np.int32)).cuda()
    dKp = dev.dzeros(N * N)
    assert lib.cxb_sym_permute_lower(None, N, dev.ptr(dK), N, dev.ptr(dperm), dev.ptr(dKp), N) == 0
    ds = dev.dzeros(N)
    work = dev.dzeros(lib.cxb_ldlt_worksize(N))
    dinfo = dev.izeros(2)
    assert lib.cxb_ldlt_lower(None, N, dev.ptr(dKp), N, dev.ptr(ds), dev.ptr(work), dev.ptr(dinfo)) == 0
    return np.tril(dev.from_dev(dKp, N, N)), dev.from_dev(ds), dinfo.cpu().tolist()[1]


def check_cholesky(H, out, info, shared=None):
    assert (info == 0).all()
    for p in range(len(H)):
        Lp = np.tril(out[p])
        assert rel(Lp, np.linalg.cholesky(H[p])) < 1e-12, p
        assert rel(Lp, single_matrix_cholesky(H[p])) < 1e-12, p
        if shared is not None:
            assert rel(Lp, np.tril(shared[p])) < 1e-12, p


def check_ldlt(K, L, perm, signs, info, Kafter, shared=None):
    assert np.array_equal(Kafter, K)
    for p in range(len(K)):
        order = rldlt_pivot_order(np.diag(K[p]))
        assert perm[p].tolist() == order == product_pivot_order(np.diag(K[p]))
        Lr, sr, reg = regularised_ldlt(K[p][np.ix_(order, order)])
        Lp = np.tril(L[p])
        assert np.array_equal(signs[p], sr) and info[p] == reg, p
        assert rel(Lp, Lr) < 1e-12, p
        Ls, ss, regs = single_matrix_ldlt(K[p], order)
        assert np.array_equal(signs[p], ss) and info[p] == regs, p
        assert rel(Lp, Ls) < 1e-12, p
        if shared is not None:
            Lsh, psh, ssh, ish = shared
            assert perm[p].tolist() == psh[p].tolist() and np.array_equal(signs[p], ssh[p]) and info[p] == ish[p]
            assert rel(Lp, np.tril(Lsh[p])) < 1e-12, p


def kkt_batch(rng, N, B=3, zero_pivot=True):
    rows = N // 4
    K = np.stack([kkt_matrix(rng, N - rows, rows) for _ in range(B)])
    if zero_pivot:
        K[1][2, :] = K[1][:, 2] = 0.0  # a zero pivot: the regularisation
    return K


@pytest.mark.parametrize("N", [1, 2, NB - 1, NB, NB + 1, 2 * NB + 3, 169])
def test_blocked_kernels_called_directly(be, N):
    """At sizes the shared-memory kernels also handle: the blocked kernels against numpy, the single-matrix path and
    the shared-memory kernels."""
    rng = np.random.Generator(np.random.PCG64(N))
    H = np.stack([spd(rng, N) for _ in range(3)])
    out, info, _ = be.potrf(H, blocked=True)
    shared, sinfo, _ = be.potrf(H, blocked=False)
    assert (sinfo == 0).all()
    check_cholesky(H, out, info, shared)
    K = kkt_batch(rng, N) if N > 4 else np.stack([spd(rng, N) - 0.5 * np.eye(N) for _ in range(3)])
    L, perm, signs, linfo, _, Kafter = be.ldlt(K, blocked=True)
    Ls, ps, ss, ls, _, _ = be.ldlt(K, blocked=False)
    check_ldlt(K, L, perm, signs, linfo, Kafter, shared=(Ls, ps, ss, ls))


@pytest.mark.parametrize("N", [171, 216, 316, 596])
def test_entry_points_above_shared_memory(be, N):
    """cxb_small_potrf / cxb_small_ldlt at sizes that used to fail: the same contract."""
    rng = np.random.Generator(np.random.PCG64(10 + N))
    B = 2
    H = np.stack([spd(rng, N) for _ in range(B)])
    out, info, _ = be.potrf(H, blocked=False)
    check_cholesky(H, out, info)
    K = kkt_batch(rng, N, B)
    L, perm, signs, linfo, _, Kafter = be.ldlt(K, blocked=False)
    check_ldlt(K, L, perm, signs, linfo, Kafter)


def test_cholesky_failure_column(be):
    rng = np.random.Generator(np.random.PCG64(77))
    N = 216
    H = np.stack([spd(rng, N) for _ in range(3)])
    for p, f in ((1, 100), (2, 171)):
        M = H[p]
        M[f, f] -= 1.0 + M[f, f] - M[f, :f] @ np.linalg.solve(M[:f, :f], M[:f, f])
    _, info, _ = be.potrf(H, blocked=False)
    assert info.tolist() == [0, 101, 172]


def test_masked_programs_are_untouched(be):
    rng = np.random.Generator(np.random.PCG64(21))
    B, N = 4, 216
    active = np.array([0, 1, 0, 1], dtype=np.int32)
    sentinel = rng.uniform(-1, 1, size=(B, N, N))
    H = np.stack([spd(rng, N) for _ in range(B)])
    out, info, _ = be.potrf(H, blocked=False, active=active, H_init=sentinel)
    K = kkt_batch(rng, N, B)
    L, perm, signs, linfo, _, Kafter = be.ldlt(K, blocked=False, active=active, L_init=sentinel)
    assert np.array_equal(Kafter, K)
    for p in range(B):
        if active[p]:
            assert info[p] == 0 and rel(np.tril(out[p]), np.linalg.cholesky(H[p])) < 1e-12
        else:
            assert np.array_equal(out[p], sentinel[p]) and info[p] == -3
            assert np.array_equal(L[p], sentinel[p]) and linfo[p] == -3
            assert (perm[p] == -7).all() and (signs[p] == 5.0).all()


def test_solves_at_large_order(be):
    """The existing one-warp solves on the blocked factors at N = 596."""
    rng = np.random.Generator(np.random.PCG64(596))
    N, B = 596, 2
    H = np.stack([spd(rng, N) for _ in range(B)])
    X = rng.uniform(-1, 1, size=(B, N))
    _, info, buf = be.potrf(H, blocked=False)
    assert (info == 0).all()
    x = be.potrs(buf, B, N, X)
    K = kkt_batch(rng, N, B, zero_pivot=False)
    _, _, _, _, handles, _ = be.ldlt(K, blocked=False)
    z = be.ldlt_solve(handles, B, N, X)
    for M, sol in ((H, x), (K, z)):
        for p in range(B):
            r = np.linalg.norm(M[p] @ sol[p] - X[p]) / (np.linalg.norm(M[p], 2) * np.linalg.norm(sol[p]))
            assert r <= 1e-10, (p, r)


# ---- whole solves -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("stages,eq_rows,kkt_order", [(22, 4, 216), (29, 0, 174), (32, 4, 316)])
def test_long_horizon_batches(libs, stages, eq_rows, kkt_order):
    O, D = libs
    gen = [mpc_problem(700 + p, stages=stages, eq_rows=eq_rows) for p in range(3)]
    probs = [(cones, b) for cones, _, b in gen]
    m = probs[0][1].size
    assert make_program(D, m, probs[0][0]).kkt_size() == kkt_order
    batch = make_batch(D, m, probs)
    solved, y = batch.maximize(np.stack([pb for _, pb in probs]), D.default_config())
    assert solved.all()
    check_both_references(O, D, m, probs, {}, batch_outcome(batch, solved, y))


def test_warm_start_after_update_at_316(libs):
    """An update of the first LP block, then a warm solve: each program as CONEX_Maximize's warm start on the old
    program's memory."""
    _, D = libs
    gen = [mpc_problem(800 + p, stages=32) for p in range(3)]
    probs = [(cones, b) for cones, _, b in gen]
    m = probs[0][1].size
    b = np.stack([pb for _, pb in probs])
    new, blocks = updated(probs, 0, 0, 3, 801, 0.01)
    warm = make_batch(D, m, probs)
    warm.maximize(b)
    warm.update(0, 0, blocks)
    solved, y = warm.maximize(b, D.default_config(initialization_mode=1))
    got = batch_outcome(warm, solved, y)
    for p, ((cones, pb), (new_cones, _)) in enumerate(zip(probs, new)):
        Q = make_program(D, m, cones)
        Q.maximize(pb)
        Q2 = D.program_on_memory_of(Q, m)
        add_cones(Q2, new_cones)
        s2, y2 = Q2.maximize(pb, D.default_config(initialization_mode=1))
        assert_parity(got[p], Q2.iteration_log(), y2, s2, tag=p)
        del Q2  # before Q: it lives on Q's memory
