"""The symmetric form of the Schur assembly reads only the lower triangle of every constraint matrix A_i and of C:
K1 forms L^T A_i L from tril(A_i) (W = L L^T), so whatever the strict upper triangle holds, NaN included, never
reaches the packed scaled matrices or the Newton system. Checked against numpy's L^T A L of the true symmetric
matrices at shapes that cover ragged 64 x 64 tiles, one and several tile rows, and panels of 1, 2 and all m + 1
matrices (batch strides of both K1 products)."""
import ctypes as C

import numpy as np
import pytest

from harness import random_sym

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    import devlib
    return devlib


def pack_lower_tiles(S):
    """numpy restatement of the packed layout: lower 64 x 64 tiles of the symmetric S, tile after tile (column of
    tiles by column of tiles), column-major inside a tile, zero-padded, off-diagonal tiles scaled by sqrt(2)."""
    n = S.shape[0]
    T = (n + 63) // 64
    P = np.zeros((T * 64, T * 64))
    P[:n, :n] = S
    out = []
    for tn in range(T):
        for tm in range(tn, T):
            tile = P[tm * 64:(tm + 1) * 64, tn * 64:(tn + 1) * 64]
            out.append((1.0 if tm == tn else np.sqrt(2.0)) * tile.ravel(order="F"))
    return np.concatenate(out)


def rel_err(x, ref):
    return np.abs(x - ref).max() / max(np.abs(ref).max(), 1e-300)


@pytest.mark.parametrize("n", [1, 17, 63, 64, 65, 193])
def test_symmetric_form_reads_only_the_lower_triangle(dev, n):
    import torch
    L = dev.product().lib
    vp = C.c_void_p
    L.cxb_packed_symmetric_size.restype = C.c_size_t
    L.cxb_packed_symmetric_size.argtypes = [C.c_int]
    L.cxb_schur_dense_lmi_sym.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp, C.c_int, vp, vp, vp, C.c_long]
    m = 3
    rng = np.random.default_rng(1000 + n)
    mats = [random_sym(rng, n) for _ in range(m)] + [random_sym(rng, n) + np.eye(n)]  # A_0 .. A_{m-1}, C
    R = rng.standard_normal((n, n))
    W = R @ R.T / n + 0.5 * np.eye(n)
    Lw = np.linalg.cholesky(W)
    upper = np.triu(np.ones((n, n), dtype=bool), 1)
    stored = []
    for A in mats:
        Au = A.copy()
        Au[upper] = np.nan
        stored.append(np.asfortranarray(Au).ravel(order="F"))
    dA = torch.from_numpy(np.concatenate(stored)).cuda()
    dW = dev.to_dev(W)

    scaled = [Lw.T @ A @ Lw for A in mats] + [np.eye(n)]  # L^T A_i L, L^T C L, I
    ref_X = [pack_lower_tiles(S) for S in scaled]
    As, Cm = mats[:m], mats[m]
    G = np.array([[np.trace(Ai @ W @ Aj @ W) for Aj in As] for Ai in As])
    AW = np.array([np.trace(Ai @ W) for Ai in As])
    AQc = np.array([np.trace(Cm @ W @ Ai @ W) for Ai in As])

    kp = L.cxb_packed_symmetric_size(n)
    ldh = (m + 3) & ~1
    for panel in (1, 2, m + 1):
        # every output and scratch buffer starts as NaN: an entry the kernels fail to write, or a scratch entry
        # they read before writing it, shows up in the result
        dX = torch.full(((m + 2) * kp,), float("nan"), dtype=torch.float64, device="cuda")
        dT = torch.full((panel * n * n,), float("nan"), dtype=torch.float64, device="cuda")
        dL = torch.full((n * n,), float("nan"), dtype=torch.float64, device="cuda")
        dH = dev.dzeros(ldh * (m + 2))
        info = dev.izeros(2)
        assert L.cxb_schur_dense_lmi_sym(None, n, m, dev.ptr(dA), dev.ptr(dW), dev.ptr(dX), dev.ptr(dT), panel,
                                         dev.ptr(dL), dev.ptr(info), dev.ptr(dH), ldh) == 0
        assert int(info.cpu()[0]) == 0
        X = dX.cpu().numpy().reshape(m + 2, kp)
        assert np.isfinite(X).all()
        for i, (S, ref) in enumerate(zip(scaled, ref_X)):
            assert np.abs(X[i] - ref).max() < 1e-11 * max(1.0, np.abs(S).max()), (panel, i)
        Haug = dev.from_dev(dH, ldh, m + 2)
        assert np.isfinite(Haug[:m + 2, :m + 1]).all()
        scale = np.sqrt(np.outer(np.diag(G), np.diag(G)))
        assert (np.abs(np.tril(Haug[:m, :m]) - np.tril(G)) / scale).max() < 1e-10
        assert rel_err(Haug[m, :m], AQc) < 1e-10
        assert rel_err(Haug[m + 1, :m], AW) < 1e-10
        assert abs(Haug[m + 1, m] - np.trace(W @ Cm)) <= 1e-10 * max(1.0, abs(np.trace(W @ Cm)))
        assert abs(Haug[m, m] - np.trace(Cm @ W @ Cm @ W)) <= 1e-10 * abs(np.trace(Cm @ W @ Cm @ W))
